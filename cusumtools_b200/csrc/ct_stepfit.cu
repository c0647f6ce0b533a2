// Batched step-response fit of events (type 1): one warp per short window, one CTA per long window.
//
// The reference consumes the result only (readevents.py:1334-1337 reads a type-1 event file with the columns
// time, current, cusum, stepfit; events.csv carries rc_const1_us / rc_const2_us); the definition of record is
// oracle/stepfit_oracle.py.  For window sample t = 0 .. n-1 and p = (i0, a, u1, u2, tau1, tau2):
//   f(t) = i0 - a (1 - exp(-(t-u1)/tau1)) H(t-u1) + a (1 - exp(-(t-u2)/tau2)) H(t-u2),   H(s) = [s >= 0]
// fitted by Levenberg-Marquardt with Marquardt scaling.  Work per trial: ONE pass over the window, which evaluates
// the trial point and leaves its cost, J^T J (21 sums) and J^T r (6 sums): an accepted trial already holds the
// normal equations of the next step, a rejected one falls back to the saved sums of the current point.
//   * the window is staged once in shared memory relative to its first sample (4 B/sample of HBM traffic); windows
//     longer than the staging slot are read from global memory (L1/L2) on every pass;
//   * per sample: float32 (two exp, ~40 FMA); per thread the 28 sums are float32, the warp reduction (a 31-shuffle
//     reduce-scatter butterfly) and the 6x6 Cholesky solve are float64;
//   * the LM state (the sums of the current point and of the trial) lives in shared memory; one thread solves, every
//     thread reads the step behind a barrier and takes the same decisions.
// The two kernels share everything but the evaluation pass (fit_window<Team>): ct_stepfit_kernel fits one window of at
// most CT_STEPFIT_MAX_WINDOW samples per warp (a Team of 32 lanes, barrier __syncwarp); ct_stepfit_long_kernel one
// window of up to CT_STEPFIT_LONG_MAX_WINDOW samples per CTA (kSfLongWarps warps whose totals are added in float64
// through shared memory, barrier __syncthreads).  oracle/stepfit_twin.py restates that shared loop.
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {

constexpr int kSfWarps = 8;                 // warps per CTA
constexpr int kSfSlot = 2048;               // samples of a window staged in shared memory (8 KB per warp)
constexpr int kSfSums = 28;                 // cost, J^T r [6], J^T J upper triangle [21]
constexpr int kSfLongWarps = 8;             // warps of the CTA that fits one long window
constexpr int kSfLongThreads = kSfLongWarps * 32;
constexpr int kSfLongSlot = 16384;          // samples of a long window staged in shared memory (64 KB per CTA)
constexpr int kSfLongClaim = 4;             // rows a CTA of the long kernel claims at a time
constexpr int kTypeAccepted = 0, kTypeStepFit = 1, kTypeStepFitFailed = 7, kTypeStepFitLong = CT_TYPE_STEPFIT_LONG;

struct StepArgs {
    const float* y; long long ntot;
    const long long* w0; const long long* w1; int* type;
    const long long* nev_dev; long long cap;
    int padding; float tau0; int max_iters; int max_levels;
    double* params; double* cost; int* iters;
    int* n_levels; int* edges; double* mean; double* sd;
};

struct FitState {
    double cur[32];                         // sums of the current point (index: kSfSums layout)
    double trial[32];                       // sums of the last evaluated trial point
    double p[8], q[8];                      // current point, trial point
    double M[24];                           // the scaled normal matrix, factorised in place (thread 0)
    double d[8];                            // the step (thread 0's solve): d[0..5], predicted decrease d[6], ok d[7]
};

struct WarpSmem {
    FitState s;
    float x[kSfSlot];                       // the window minus its first sample
};

struct LongSmem {
    FitState s;
    double red[kSfLongWarps * 32];          // per-warp totals of the evaluation pass (warp w: red[32 w .. 32 w + 28))
    double tot[kSfLongWarps];               // per-warp totals of a scalar sum
    long long claim;                        // the first of the rows the CTA claimed last
    float x[kSfLongSlot];                   // the window minus its first sample
};

// a model point in the form the per-sample loop consumes: the window frame (i0 relative to x[0]), the step positions
// split into an integer part and a fraction in [0, 1) so that H(t - u) is decided exactly as in float64
struct ModelF {
    float i0, a, it1, it2, fr1, fr2;
    int k1, k2;
};

__device__ __forceinline__ ModelF model_point(const double* p) {
    ModelF m;
    m.i0 = (float)p[0]; m.a = (float)p[1];
    const double f1 = floor(p[2]), f2 = floor(p[3]);
    m.k1 = (int)f1; m.k2 = (int)f2;
    // rounded up: a fraction that is not 0 in float64 must not become 0 (H at t == k); kept below 1
    m.fr1 = fminf(__double2float_ru(p[2] - f1), 0.99999994f);
    m.fr2 = fminf(__double2float_ru(p[3] - f2), 0.99999994f);
    m.it1 = (float)(1.0 / p[4]); m.it2 = (float)(1.0 / p[5]);
    return m;
}

// sum over the 32 lanes of 32 per-lane float32 values in float64: lane L ends with the total of index L (a reduce-scatter
// butterfly, 31 shuffles; the first round converts, so at most 16 float64 partial sums are live)
__device__ __forceinline__ double reduce_scatter32(const float (&f)[32], int lane) {
    double v[16];
    {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const double send = up ? f[i] : f[i + 16];
            const double keep = up ? f[i + 16] : f[i];
            v[i] = keep + __shfl_xor_sync(CT_FULL, send, 16);
        }
    }
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1) {
        const bool up = (lane & w) != 0;
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const double send = up ? v[i] : v[i + w];
            const double keep = up ? v[i + w] : v[i];
            v[i] = keep + __shfl_xor_sync(CT_FULL, send, w);
        }
    }
    return v[0];
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CT_FULL, v, o);
    return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(CT_FULL, v, o));
    return v;
}

// One thread's pass over its samples t = first, first + stride, ...: cost, J^T r and J^T J of the model point `p` into
// acc (float32: cost, J^T r [6], J^T J [21], 4 unused)
__device__ __forceinline__ void accumulate(const float* __restrict__ src, float xoff, int n, const double* p, int first,
                                           int stride, float (&acc)[32]) {
    const ModelF m = model_point(p);
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    float& c = acc[0];
    float* g = acc + 1;
    float* A = acc + 7;
    for (int t = first; t < n; t += stride) {
        const float x = src[t] - xoff;
        const float s1 = (float)(t - m.k1) - m.fr1, s2 = (float)(t - m.k2) - m.fr2;
        const bool h1 = s1 >= 0.f, h2 = s2 >= 0.f;
        const float e1 = h1 ? __expf(-s1 * m.it1) : 0.f;     // (the discarded branch may overflow: it is not used)
        const float e2 = h2 ? __expf(-s2 * m.it2) : 0.f;
        const float q1 = h1 ? 1.f - e1 : 0.f, q2 = h2 ? 1.f - e2 : 0.f;
        const float f = fmaf(m.a, q2 - q1, m.i0);
        const float r = x - f;
        float J[6];
        J[0] = 1.f;
        J[1] = q2 - q1;
        J[2] = m.a * e1 * m.it1;                 // df/du1
        J[3] = -(m.a * e2 * m.it2);              // df/du2
        J[4] = J[2] * (s1 * m.it1);              // df/dtau1 = a e1 s1 / tau1^2
        J[5] = J[3] * (s2 * m.it2);              // df/dtau2
        c = fmaf(r, r, c);
#pragma unroll
        for (int j = 0; j < 6; ++j) g[j] = fmaf(J[j], r, g[j]);
        int k = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = i; j < 6; ++j) { A[k] = fmaf(J[i], J[j], A[k]); ++k; }
    }
}

// Sum of squared residuals of the fitted model `p` over the three level rows [0, b1), [b1, b2), [b2, n) (float32 per
// thread)
__device__ __forceinline__ void level_residuals(const float* __restrict__ src, float xoff, int n, const double* p, int first,
                                                int stride, int b1, int b2, float& r0, float& r1, float& r2) {
    const ModelF m = model_point(p);
    for (int t = first; t < n; t += stride) {
        const float x = src[t] - xoff;
        const float s1 = (float)(t - m.k1) - m.fr1, s2 = (float)(t - m.k2) - m.fr2;
        const float q1 = s1 >= 0.f ? 1.f - __expf(-s1 * m.it1) : 0.f;
        const float q2 = s2 >= 0.f ? 1.f - __expf(-s2 * m.it2) : 0.f;
        const float r = x - fmaf(m.a, q2 - q1, m.i0);
        if (t < b1) r0 = fmaf(r, r, r0); else if (t < b2) r1 = fmaf(r, r, r1); else r2 = fmaf(r, r, r2);
    }
}

// The threads that fit one window.  rank: index in the team; sync(): barrier of the team; sum / max: the team's total
// of one value per thread, returned to every thread; evaluate: one pass into out[0 .. kSfSums) (shared memory).
struct WarpTeam {
    static constexpr int size = 32;
    int rank;
    __device__ void sync() const { __syncwarp(); }
    __device__ double sum(double v) const { return warp_sum(v); }
    __device__ float max(float v) const { return warp_max(v); }
    __device__ void evaluate(const float* __restrict__ src, float xoff, int n, const double* p, double* out) const {
        float acc[32];
        accumulate(src, xoff, n, p, rank, 32, acc);
        const double s = reduce_scatter32(acc, rank);
        __syncwarp();
        if (rank < kSfSums) out[rank] = s;
        __syncwarp();
    }
};

struct CtaTeam {
    static constexpr int size = kSfLongThreads;
    int rank;
    LongSmem* sm;
    __device__ void sync() const { __syncthreads(); }
    // warp totals by butterfly, then the kSfLongWarps totals in warp order (float64, the same order in every thread)
    __device__ double sum(double v) const {
        v = warp_sum(v);
        if ((rank & 31) == 0) sm->tot[rank >> 5] = v;
        __syncthreads();
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kSfLongWarps; ++w) t += sm->tot[w];
        __syncthreads();
        return t;
    }
    __device__ float max(float v) const {
        v = warp_max(v);
        if ((rank & 31) == 0) sm->tot[rank >> 5] = (double)v;
        __syncthreads();
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kSfLongWarps; ++w) t = fmax(t, sm->tot[w]);
        __syncthreads();
        return (float)t;                                // exact: the values are float32 and >= 0
    }
    __device__ void evaluate(const float* __restrict__ src, float xoff, int n, const double* p, double* out) const {
        float acc[32];
        accumulate(src, xoff, n, p, rank, kSfLongThreads, acc);
        const int lane = rank & 31, w = rank >> 5;
        const double s = reduce_scatter32(acc, lane);
        if (lane < kSfSums) sm->red[w * 32 + lane] = s;
        __syncthreads();
        if (rank < kSfSums) {
            double t = 0.0;
#pragma unroll
            for (int k = 0; k < kSfLongWarps; ++k) t += sm->red[k * 32 + rank];
            out[rank] = t;
        }
        __syncthreads();
    }
};

__device__ __forceinline__ int tri(int i, int j) {      // index of (i, j), i <= j, in the upper triangle
    return i * 6 - i * (i - 1) / 2 + (j - i);
}

// Marquardt-scaled LM step from the sums `S` of the current point: solves (A + mu diag(A)) d = g on the Jacobi-scaled
// matrix (unit diagonal) by Cholesky, in the team's shared memory (one thread; the matrix is not kept in registers).
// out[0..5] = d, out[6] = decrease of the sum of squares the linear model predicts (2 d.g - d^T A d), out[7] = 1 if
// the matrix is positive definite (0: no step).
__device__ __noinline__ void lm_step(const double* S, double mu, double* M, double* out) {
    double sc[6];
    out[7] = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double aii = S[7 + tri(i, i)];
        if (!(aii > 0.0)) return;
        sc[i] = 1.0 / sqrt(aii);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = i + 1; j < 6; ++j) M[tri(i, j)] = S[7 + tri(i, j)] * sc[i] * sc[j];
        M[tri(i, i)] = 1.0 + mu;
        out[i] = S[1 + i] * sc[i];                     // right-hand side, overwritten by the solution
    }
    // Cholesky M = R^T R, R upper triangular, in place
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double dii = M[tri(i, i)];
#pragma unroll
        for (int k = 0; k < i; ++k) dii -= M[tri(k, i)] * M[tri(k, i)];
        if (!(dii > 0.0)) return;
        const double rii = sqrt(dii);
        M[tri(i, i)] = rii;
#pragma unroll
        for (int j = i + 1; j < 6; ++j) {
            double v = M[tri(i, j)];
#pragma unroll
            for (int k = 0; k < i; ++k) v -= M[tri(k, i)] * M[tri(k, j)];
            M[tri(i, j)] = v / rii;
        }
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {                      // R^T z = b
        double v = out[i];
#pragma unroll
        for (int k = 0; k < i; ++k) v -= M[tri(k, i)] * out[k];
        out[i] = v / M[tri(i, i)];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {                     // R d' = z
        double v = out[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) v -= M[tri(i, k)] * out[k];
        out[i] = v / M[tri(i, i)];
    }
    double dAd = 0.0, dg = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) out[i] *= sc[i];       // back to parameter units
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        dg += out[i] * S[1 + i];
        double row = 0.0;
#pragma unroll
        for (int j = 0; j < 6; ++j) row += out[j] * S[7 + (i <= j ? tri(i, j) : tri(j, i))];
        dAd += out[i] * row;
    }
    out[6] = 2.0 * dg - dAd;
    out[7] = 1.0;
}

// A window the kernels do not fit (outside [0, n_total), not longer than 2 padding, longer than the kernel's limit):
// type 7 with zero params, cost and iters and no level rows (edge row -1), as a failed fit
template <class Team>
__device__ __forceinline__ void reject_window(const Team& tm, const StepArgs& a, long long ev) {
    double* prow = a.params + ev * 6;
    int* ed = a.edges + ev * (a.max_levels + 1);
    if (tm.rank < 6) prow[tm.rank] = 0.0;
    if (tm.rank == 0) { a.cost[ev] = 0.0; a.iters[ev] = 0; a.n_levels[ev] = 0; a.type[ev] = kTypeStepFitFailed; }
    for (int i = tm.rank; i <= a.max_levels; i += Team::size) ed[i] = -1;
}

// The fit of one window of n samples, src[t] - xoff = y[win_start + t] - x0 (staged, xoff = 0, or read from global
// memory, xoff = x0): initial guess, LM loop, validity, the params / cost / iters row and the level rows of row ev.
template <class Team>
__device__ __forceinline__ void fit_window(const Team& tm, const StepArgs& a, long long ev, FitState& sm,
                                           const float* __restrict__ src, float xoff, int n, float x0) {
    const int rank = tm.rank;
    const int pad = a.padding;
    double* prow = a.params + ev * 6;
    int* ed = a.edges + ev * (a.max_levels + 1);
    // ---- initial guess: i0 = mean of the 2*padding baseline samples, a = i0 - mean of the event interior
    double sb = 0.0, si = 0.0;
    float xs = 0.f;                                    // largest |x - x[0]|: the float32 resolution of the samples
    for (int t = rank; t < n; t += Team::size) {
        const float xf = src[t] - xoff;
        const double x = (double)xf;
        xs = fmaxf(xs, fabsf(xf));
        if (t < pad || t >= n - pad) sb += x; else si += x;
    }
    sb = tm.sum(sb); si = tm.sum(si); xs = tm.max(xs);
    // a cost change below n (2^-24 max|x|)^2 is below what the float32 residuals resolve: it counts as no decrease
    const double floor_ = (double)n * ((double)xs * 5.96e-8) * ((double)xs * 5.96e-8);
    const double i0_init = sb / (2.0 * pad), base_abs = (double)x0 + i0_init;
    double* p = sm.p;                                  // current and trial point in shared memory: every thread reads them
    double* q = sm.q;
    if (rank == 0) {
        p[0] = i0_init; p[1] = i0_init - si / (double)(n - 2 * pad); p[2] = (double)pad; p[3] = (double)(n - pad);
        p[4] = (double)a.tau0; p[5] = (double)a.tau0;
    }
    tm.sync();
    tm.evaluate(src, xoff, n, p, sm.cur);
    int it = 1;
    double mu = 1e-3;                                  // 1e-3 x the largest diagonal entry of the scaled matrix (1)
    bool converged = false;
    while (it < a.max_iters && mu < 1e30) {
        tm.sync();                                     // every thread has read the previous step
        if (rank == 0) lm_step(sm.cur, mu, sm.M, sm.d);
        tm.sync();
        const double* d = sm.d;
        const double pred = d[6];
        if (d[7] == 0.0) { mu *= 10.0; ++it; continue; }
        const double c = sm.cur[0];
        // the decrease the step predicts stands in for the actual one near the optimum, where float32 samples cannot
        // resolve a change of 1e-9 of the cost
        if (!(pred > 1e-9 * c + floor_)) { converged = true; break; }
        double big = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) big = fmax(big, fabs(d[i]) / (fabs(i == 0 ? p[0] + (double)x0 : p[i]) + 1e-8));
        if (big < 1e-8) { converged = true; break; }  // relative step below 1e-8
        tm.sync();
        if (rank == 0) {
#pragma unroll
            for (int i = 0; i < 6; ++i) q[i] = p[i] + d[i];
        }
        tm.sync();
        if (!(q[4] > 0.0) || !(q[5] > 0.0) || !(q[2] < q[3])) { mu *= 10.0; ++it; continue; }   // not evaluated
        tm.evaluate(src, xoff, n, q, sm.trial);
        ++it;
        const double ct = sm.trial[0];
        if (ct < c) {                                  // (a NaN cost is rejected here)
            if (rank < kSfSums) sm.cur[rank] = sm.trial[rank];
            if (rank < 6) p[rank] = q[rank];
            tm.sync();
            mu *= 0.1;
            if (c - ct < 1e-9 * c + floor_) { converged = true; break; }
        } else {
            mu *= 10.0;
        }
    }
    tm.sync();
    // ---- validity: every level row holds a sample, rise times within [0.05, n], the step in the blockage direction
    const double e1 = ceil(p[2]), e2 = ceil(p[3]);
    const bool sign_ok = base_abs >= 0.0 ? p[1] > 0.0 : p[1] < 0.0;
    const bool ok = converged && p[2] > 0.0 && e1 < e2 && e2 < (double)n && p[4] >= 0.05 && p[4] <= (double)n &&
                    p[5] >= 0.05 && p[5] <= (double)n && sign_ok;
    if (rank == 0) {
        prow[0] = p[0] + (double)x0;
#pragma unroll
        for (int i = 1; i < 6; ++i) prow[i] = p[i];
        a.cost[ev] = sm.cur[0];
        a.iters[ev] = it;
    }
    if (!ok) {
        if (rank == 0) { a.n_levels[ev] = 0; a.type[ev] = kTypeStepFitFailed; }
        for (int i = rank; i <= a.max_levels; i += Team::size) ed[i] = -1;
        return;
    }
    // ---- level rows: [0, ceil u1), [ceil u1, ceil u2), [ceil u2, n); std = rms of x - f over each
    const int b1 = (int)e1, b2 = (int)e2;
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    level_residuals(src, xoff, n, p, rank, Team::size, b1, b2, r0, r1, r2);
    const double d0 = tm.sum(r0), d1 = tm.sum(r1), d2 = tm.sum(r2);
    for (int i = rank; i <= a.max_levels; i += Team::size) ed[i] = -1;
    tm.sync();
    if (rank == 0) {
        CT_CHECK_RANGE(ev * (a.max_levels + 1), 4, a.cap * (a.max_levels + 1), "stepfit, edge row");
        CT_CHECK_RANGE(ev * a.max_levels, 3, a.cap * a.max_levels, "stepfit, level row");
        ed[0] = 0; ed[1] = b1; ed[2] = b2; ed[3] = n;
        const double i0 = p[0] + (double)x0;
        double* mu_ = a.mean + ev * a.max_levels;
        double* sd_ = a.sd + ev * a.max_levels;
        mu_[0] = i0; mu_[1] = i0 - p[1]; mu_[2] = i0;
        sd_[0] = sqrt(d0 / b1); sd_[1] = sqrt(d1 / (b2 - b1)); sd_[2] = sqrt(d2 / (n - b2));
        a.n_levels[ev] = 3;
        a.type[ev] = kTypeStepFit;                     // (the long kernel's rows were CT_TYPE_STEPFIT_LONG)
    }
}

__device__ __forceinline__ long long event_count(const long long* nev_dev, long long cap) {
    long long nev = cap;
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    return nev;
}

__global__ void __launch_bounds__(kSfWarps * 32) ct_stepfit_select_kernel(const long long* __restrict__ w0,
                                                                           const long long* __restrict__ w1,
                                                                           int* __restrict__ type,
                                                                           const long long* __restrict__ nev_dev,
                                                                           long long cap, long long padding, long long samples) {
    const long long nev = event_count(nev_dev, cap);
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x) {
        if (type[ev] == kTypeAccepted && w1[ev] - w0[ev] - 2 * padding < samples) type[ev] = kTypeStepFit;
    }
}

__global__ void __launch_bounds__(256) ct_stepfit_fallback_select_kernel(const int* __restrict__ n_levels,
                                                                         const unsigned char* __restrict__ overflow,
                                                                         const long long* __restrict__ w0,
                                                                         const long long* __restrict__ w1,
                                                                         int* __restrict__ type,
                                                                         const long long* __restrict__ nev_dev, long long cap) {
    const long long nev = event_count(nev_dev, cap);
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x) {
        if (type[ev] == kTypeAccepted && overflow[ev] == 0 && n_levels[ev] < 3)
            type[ev] = w1[ev] - w0[ev] <= CT_STEPFIT_MAX_WINDOW ? kTypeStepFit : kTypeStepFitLong;
    }
}

__global__ void __launch_bounds__(kSfWarps * 32, 2) ct_stepfit_kernel(StepArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = ct_lane(), wib = threadIdx.x >> 5;
    WarpSmem& sm = reinterpret_cast<WarpSmem*>(smem_raw)[wib];
    const long long nev = event_count(a.nev_dev, a.cap);
    const long long ev = (long long)blockIdx.x * kSfWarps + wib;
    if (ev >= nev) return;
    if (a.type[ev] != kTypeStepFit) {                  // rows of other events: zero (their level rows are not ours)
        double* prow = a.params + ev * 6;
        if (lane < 6) prow[lane] = 0.0;
        if (lane == 0) { a.cost[ev] = 0.0; a.iters[ev] = 0; }
        return;
    }
    const WarpTeam tm{lane};
    const long long p0 = a.w0[ev], p1 = a.w1[ev];
    const long long nn = p1 - p0;
    if (p0 < 0 || p1 > a.ntot || nn <= 2LL * a.padding || nn > CT_STEPFIT_MAX_WINDOW) {
        reject_window(tm, a, ev);
        return;
    }
    const int n = (int)nn;
    const float x0 = a.y[p0];
    const float* src;
    float xoff;
    if (n <= kSfSlot) {
        for (int t = lane; t < n; t += 32) sm.x[t] = a.y[p0 + t] - x0;
        src = sm.x; xoff = 0.f;
    } else {
        src = a.y + p0; xoff = x0;
    }
    __syncwarp();
    fit_window(tm, a, ev, sm.s, src, xoff, n, x0);
}

// One long window: staged (up to kSfLongSlot samples) or read from global memory, then fitted by the whole CTA
__device__ __forceinline__ void fit_long_row(const CtaTeam& tm, const StepArgs& a, LongSmem& sm, long long ev) {
    const long long p0 = a.w0[ev], p1 = a.w1[ev];
    const long long nn = p1 - p0;
    if (p0 < 0 || p1 > a.ntot || nn <= 2LL * a.padding || nn > CT_STEPFIT_LONG_MAX_WINDOW) {
        if (threadIdx.x == 0) CT_CHECK_RANGE(ev, 1, a.cap, "stepfit long, rejected row");
        reject_window(tm, a, ev);
        return;
    }
    const int n = (int)nn;
    const float x0 = a.y[p0];
    const float* src;
    float xoff;
    if (n <= kSfLongSlot) {
        if (threadIdx.x == 0) CT_CHECK_RANGE(0, n, kSfLongSlot, "stepfit long, staging slot");
        for (int t = threadIdx.x; t < n; t += kSfLongThreads) sm.x[t] = a.y[p0 + t] - x0;
        src = sm.x; xoff = 0.f;
    } else {
        src = a.y + p0; xoff = x0;
    }
    __syncthreads();
    fit_window(tm, a, ev, sm.s, src, xoff, n, x0);
}

// One CTA per long window.  The resident CTAs claim the rows kSfLongClaim at a time from a counter in device memory
// (rows differ in cost by more than 10x: a static assignment lets a periodic trace give some CTAs all the longest
// windows) and fit the claimed rows of type CT_TYPE_STEPFIT_LONG.  Every other row is left as it is; a row's result
// does not depend on which CTA fits it.
__global__ void __launch_bounds__(kSfLongThreads, 2) ct_stepfit_long_kernel(StepArgs a, unsigned long long* counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    LongSmem& sm = *reinterpret_cast<LongSmem*>(smem_raw);
    const CtaTeam tm{(int)threadIdx.x, &sm};
    const long long nev = event_count(a.nev_dev, a.cap);
    for (;;) {
        __syncthreads();                               // the previous rows are done with the shared memory
        if (threadIdx.x == 0) sm.claim = (long long)atomicAdd(counter, (unsigned long long)kSfLongClaim);
        __syncthreads();
        const long long base = sm.claim;
        if (base >= nev) break;
        unsigned todo = 0;                             // bit j: row base + j is of type CT_TYPE_STEPFIT_LONG
#pragma unroll
        for (int j = 0; j < kSfLongClaim; ++j)
            if (base + j < nev && a.type[base + j] == kTypeStepFitLong) todo |= 1u << j;
        __syncthreads();                               // every thread has read the types before thread 0 may change one
        while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1;
            __syncthreads();                           // the previous row is done with the shared memory
            fit_long_row(tm, a, sm, base + j);
        }
    }
}

}  // namespace

extern "C" int ct_stepfit_select(const int64_t* win_start, const int64_t* win_end, int32_t* type, const int64_t* n_events_dev,
                                 int64_t capacity, int64_t padding, int64_t stepfit_samples, void* stream) {
    if (!win_start || !win_end || !type || capacity < 0 || padding < 0) { ct_set_error("stepfit_select: bad argument"); return CT_ERR_ARG; }
    if (capacity == 0 || stepfit_samples <= 0) return CT_OK;
    long long grid = (capacity + 255) / 256;
    const long long lim = (long long)ct_sm_count() * 8;
    if (grid > lim) grid = lim;
    CT_COUNT_LAUNCH();
    ct_stepfit_select_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        (const long long*)win_start, (const long long*)win_end, type, (const long long*)n_events_dev, capacity, padding,
        stepfit_samples);
    return ct_check_launch("ct_stepfit_select_kernel");
}

extern "C" int ct_stepfit_fallback_select(const int32_t* n_levels, const uint8_t* overflow, const int64_t* win_start,
                                          const int64_t* win_end, int32_t* type, const int64_t* n_events_dev, int64_t capacity,
                                          void* stream) {
    if (!n_levels || !overflow || !win_start || !win_end || !type || capacity < 0) {
        ct_set_error("stepfit_fallback_select: bad argument"); return CT_ERR_ARG;
    }
    if (capacity == 0) return CT_OK;
    long long grid = (capacity + 255) / 256;
    const long long lim = (long long)ct_sm_count() * 8;
    if (grid > lim) grid = lim;
    CT_COUNT_LAUNCH();
    ct_stepfit_fallback_select_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        n_levels, overflow, (const long long*)win_start, (const long long*)win_end, type, (const long long*)n_events_dev,
        capacity);
    return ct_check_launch("ct_stepfit_fallback_select_kernel");
}

namespace {

int stepfit_args(StepArgs& a, const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end, int32_t* type,
                 const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0, int max_iters, int max_levels,
                 double* params6, double* cost, int32_t* iters, int32_t* n_levels, int32_t* edges, double* level_mean,
                 double* level_std, int64_t max_window) {
    if (!y || !win_start || !win_end || !type || !params6 || !cost || !iters || !n_levels || !edges || !level_mean || !level_std) {
        ct_set_error("stepfit: null pointer"); return CT_ERR_ARG;
    }
    if (capacity < 0 || padding < 1 || padding > max_window || !(tau0 > 0.f) || max_iters < 1 || max_levels < 3) {
        ct_set_error("stepfit: bad argument (need padding >= 1, tau0 > 0, max_iters >= 1, max_levels >= 3)"); return CT_ERR_ARG;
    }
    a.y = y; a.ntot = n_total; a.w0 = (const long long*)win_start; a.w1 = (const long long*)win_end; a.type = type;
    a.nev_dev = (const long long*)n_events_dev; a.cap = capacity; a.padding = (int)padding; a.tau0 = tau0;
    a.max_iters = max_iters; a.max_levels = max_levels; a.params = params6; a.cost = cost; a.iters = iters;
    a.n_levels = n_levels; a.edges = edges; a.mean = level_mean; a.sd = level_std;
    return CT_OK;
}

}  // namespace

extern "C" int ct_stepfit_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end, int32_t* type,
                                const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0, int max_iters,
                                int max_levels, double* params6, double* cost, int32_t* iters, int32_t* n_levels, int32_t* edges,
                                double* level_mean, double* level_std, void* stream) {
    StepArgs a;
    const int rc = stepfit_args(a, y, n_total, win_start, win_end, type, n_events_dev, capacity, padding, tau0, max_iters,
                                max_levels, params6, cost, iters, n_levels, edges, level_mean, level_std, CT_STEPFIT_MAX_WINDOW);
    if (rc != CT_OK) return rc;
    if (capacity == 0) return CT_OK;
    if (capacity > 0x7fffffffLL * kSfWarps) { ct_set_error("stepfit: too many events in one batch"); return CT_ERR_UNSUPPORTED; }
    const int smem = kSfWarps * (int)sizeof(WarpSmem);
    if (cudaFuncSetAttribute(ct_stepfit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
        ct_set_error("stepfit: cannot reserve %d bytes of shared memory", smem); return CT_ERR_CUDA;
    }
    const long long grid = (capacity + kSfWarps - 1) / kSfWarps;
    CT_COUNT_LAUNCH();
    ct_stepfit_kernel<<<(unsigned)grid, kSfWarps * 32, smem, (cudaStream_t)stream>>>(a);
    return ct_check_launch("ct_stepfit_kernel");
}

extern "C" int ct_stepfit_long_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                                     int32_t* type, const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0,
                                     int max_iters, int max_levels, double* params6, double* cost, int32_t* iters,
                                     int32_t* n_levels, int32_t* edges, double* level_mean, double* level_std,
                                     int64_t* row_counter, void* stream) {
    if (!row_counter) { ct_set_error("stepfit long: null row counter"); return CT_ERR_ARG; }
    StepArgs a;
    const int rc = stepfit_args(a, y, n_total, win_start, win_end, type, n_events_dev, capacity, padding, tau0, max_iters,
                                max_levels, params6, cost, iters, n_levels, edges, level_mean, level_std,
                                CT_STEPFIT_LONG_MAX_WINDOW);
    if (rc != CT_OK) return rc;
    if (capacity == 0) return CT_OK;
    const int smem = (int)sizeof(LongSmem);
    if (cudaFuncSetAttribute(ct_stepfit_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
        ct_set_error("stepfit long: cannot reserve %d bytes of shared memory", smem); return CT_ERR_CUDA;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ct_stepfit_long_kernel, kSfLongThreads, smem) != cudaSuccess ||
        per_sm < 1) {
        ct_set_error("stepfit long: the kernel does not fit on a multiprocessor"); return CT_ERR_CUDA;
    }
    long long grid = (long long)ct_sm_count() * per_sm;   // resident CTAs; each claims rows until none is left
    const long long claims = (capacity + kSfLongClaim - 1) / kSfLongClaim;
    if (grid > claims) grid = claims;
    if (cudaMemsetAsync(row_counter, 0, sizeof(int64_t), (cudaStream_t)stream) != cudaSuccess) {
        ct_set_error("stepfit long: cannot reset the row counter"); return CT_ERR_CUDA;
    }
    CT_COUNT_LAUNCH();
    ct_stepfit_long_kernel<<<(unsigned)grid, kSfLongThreads, smem, (cudaStream_t)stream>>>(
        a, reinterpret_cast<unsigned long long*>(row_counter));
    return ct_check_launch("ct_stepfit_long_kernel");
}
