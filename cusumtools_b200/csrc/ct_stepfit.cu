// Batched step-response fit of short events (type 1), one warp per event.
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
//   * per sample: float32 (two exp, ~40 FMA); per lane the 28 sums are float32, the warp reduction (a 31-shuffle
//     reduce-scatter butterfly) and the 6x6 Cholesky solve are float64;
//   * the LM state (the sums of the current point and of the trial) lives in shared memory; every lane runs the same
//     float64 solve, so the warp stays convergent and no lane has to broadcast a decision.
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {

constexpr int kSfWarps = 8;                 // warps per CTA
constexpr int kSfSlot = 2048;               // samples of a window staged in shared memory (8 KB per warp)
constexpr int kSfSums = 28;                 // cost, J^T r [6], J^T J upper triangle [21]
constexpr int kTypeAccepted = 0, kTypeStepFit = 1, kTypeStepFitFailed = 7;

struct StepArgs {
    const float* y; long long ntot;
    const long long* w0; const long long* w1; int* type;
    const long long* nev_dev; long long cap;
    int padding; float tau0; int max_iters; int max_levels;
    double* params; double* cost; int* iters;
    int* n_levels; int* edges; double* mean; double* sd;
};

struct WarpSmem {
    double cur[32];                         // sums of the current point (index: kSfSums layout)
    double trial[32];                       // sums of the last evaluated trial point
    double p[8], q[8];                      // current point, trial point
    double M[24];                           // the scaled normal matrix, factorised in place (lane 0)
    double d[8];                            // the step (lane 0's solve): d[0..5], predicted decrease d[6], ok d[7]
    float x[kSfSlot];                       // the window minus its first sample
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

// One pass: cost, J^T r and J^T J of the model point `p` over the window into out[0 .. kSfSums) (shared memory).
__device__ __forceinline__ void evaluate(const float* __restrict__ src, float xoff, int n, const double* p, int lane, double* out) {
    const ModelF m = model_point(p);
    float acc[32];                               // cost, J^T r [6], J^T J [21], 4 unused
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    float& c = acc[0];
    float* g = acc + 1;
    float* A = acc + 7;
    for (int t = lane; t < n; t += 32) {
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
    const double s = reduce_scatter32(acc, lane);
    __syncwarp();
    if (lane < kSfSums) out[lane] = s;
    __syncwarp();
}

__device__ __forceinline__ int tri(int i, int j) {      // index of (i, j), i <= j, in the upper triangle
    return i * 6 - i * (i - 1) / 2 + (j - i);
}

// Marquardt-scaled LM step from the sums `S` of the current point: solves (A + mu diag(A)) d = g on the Jacobi-scaled
// matrix (unit diagonal) by Cholesky, in the warp's shared memory (one lane; the matrix is not kept in registers).
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

__global__ void __launch_bounds__(kSfWarps * 32) ct_stepfit_select_kernel(const long long* __restrict__ w0,
                                                                           const long long* __restrict__ w1,
                                                                           int* __restrict__ type,
                                                                           const long long* __restrict__ nev_dev,
                                                                           long long cap, long long padding, long long samples) {
    long long nev = cap;
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x) {
        if (type[ev] == kTypeAccepted && w1[ev] - w0[ev] - 2 * padding < samples) type[ev] = kTypeStepFit;
    }
}

__global__ void __launch_bounds__(kSfWarps * 32, 2) ct_stepfit_kernel(StepArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = ct_lane(), wib = threadIdx.x >> 5;
    WarpSmem& sm = reinterpret_cast<WarpSmem*>(smem_raw)[wib];
    long long nev = a.cap;
    if (a.nev_dev) { const long long d = *a.nev_dev; nev = d < nev ? d : nev; }
    const long long ev = (long long)blockIdx.x * kSfWarps + wib;
    if (ev >= nev) return;
    double* prow = a.params + ev * 6;
    if (a.type[ev] != kTypeStepFit) {                  // rows of other events: zero (their level rows are not ours)
        if (lane < 6) prow[lane] = 0.0;
        if (lane == 0) { a.cost[ev] = 0.0; a.iters[ev] = 0; }
        return;
    }
    const long long p0 = a.w0[ev], p1 = a.w1[ev];
    const int pad = a.padding;
    const long long nn = p1 - p0;
    int* ed = a.edges + ev * (a.max_levels + 1);
    if (p0 < 0 || p1 > a.ntot || nn <= 2LL * pad || nn > CT_STEPFIT_MAX_WINDOW) {
        if (lane < 6) prow[lane] = 0.0;
        if (lane == 0) { a.cost[ev] = 0.0; a.iters[ev] = 0; a.n_levels[ev] = 0; a.type[ev] = kTypeStepFitFailed; }
        for (int i = lane; i <= a.max_levels; i += 32) ed[i] = -1;   // as a failed fit: no level rows
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
    // ---- initial guess: i0 = mean of the 2*padding baseline samples, a = i0 - mean of the event interior
    double sb = 0.0, si = 0.0;
    float xs = 0.f;                                    // largest |x - x[0]|: the float32 resolution of the samples
    for (int t = lane; t < n; t += 32) {
        const float xf = src[t] - xoff;
        const double x = (double)xf;
        xs = fmaxf(xs, fabsf(xf));
        if (t < pad || t >= n - pad) sb += x; else si += x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sb += __shfl_xor_sync(CT_FULL, sb, o); si += __shfl_xor_sync(CT_FULL, si, o);
        xs = fmaxf(xs, __shfl_xor_sync(CT_FULL, xs, o));
    }
    // a cost change below n (2^-24 max|x|)^2 is below what the float32 residuals resolve: it counts as no decrease
    const double floor_ = (double)n * ((double)xs * 5.96e-8) * ((double)xs * 5.96e-8);
    const double i0_init = sb / (2.0 * pad), base_abs = (double)x0 + i0_init;
    double* p = sm.p;                                  // current and trial point in shared memory: every lane reads them
    double* q = sm.q;
    if (lane == 0) {
        p[0] = i0_init; p[1] = i0_init - si / (double)(n - 2 * pad); p[2] = (double)pad; p[3] = (double)(n - pad);
        p[4] = (double)a.tau0; p[5] = (double)a.tau0;
    }
    __syncwarp();
    evaluate(src, xoff, n, p, lane, sm.cur);
    int it = 1;
    double mu = 1e-3;                                  // 1e-3 x the largest diagonal entry of the scaled matrix (1)
    bool converged = false;
    while (it < a.max_iters && mu < 1e30) {
        __syncwarp();                                  // every lane has read the previous step
        if (lane == 0) lm_step(sm.cur, mu, sm.M, sm.d);
        __syncwarp();
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
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 6; ++i) q[i] = p[i] + d[i];
        }
        __syncwarp();
        if (!(q[4] > 0.0) || !(q[5] > 0.0) || !(q[2] < q[3])) { mu *= 10.0; ++it; continue; }   // not evaluated
        evaluate(src, xoff, n, q, lane, sm.trial);
        ++it;
        const double ct = sm.trial[0];
        if (ct < c) {                                  // (a NaN cost is rejected here)
            if (lane < kSfSums) sm.cur[lane] = sm.trial[lane];
            if (lane < 6) p[lane] = q[lane];
            __syncwarp();
            mu *= 0.1;
            if (c - ct < 1e-9 * c + floor_) { converged = true; break; }
        } else {
            mu *= 10.0;
        }
    }
    __syncwarp();
    // ---- validity: every level row holds a sample, rise times within [0.05, n], the step in the blockage direction
    const double e1 = ceil(p[2]), e2 = ceil(p[3]);
    const bool sign_ok = base_abs >= 0.0 ? p[1] > 0.0 : p[1] < 0.0;
    const bool ok = converged && p[2] > 0.0 && e1 < e2 && e2 < (double)n && p[4] >= 0.05 && p[4] <= (double)n &&
                    p[5] >= 0.05 && p[5] <= (double)n && sign_ok;
    if (lane == 0) {
        prow[0] = p[0] + (double)x0;
#pragma unroll
        for (int i = 1; i < 6; ++i) prow[i] = p[i];
        a.cost[ev] = sm.cur[0];
        a.iters[ev] = it;
    }
    if (!ok) {
        if (lane == 0) { a.n_levels[ev] = 0; a.type[ev] = kTypeStepFitFailed; }
        for (int i = lane; i <= a.max_levels; i += 32) ed[i] = -1;
        return;
    }
    // ---- level rows: [0, ceil u1), [ceil u1, ceil u2), [ceil u2, n); std = rms of x - f over each
    const int b1 = (int)e1, b2 = (int)e2;
    const ModelF m = model_point(p);
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    for (int t = lane; t < n; t += 32) {
        const float x = src[t] - xoff;
        const float s1 = (float)(t - m.k1) - m.fr1, s2 = (float)(t - m.k2) - m.fr2;
        const float q1 = s1 >= 0.f ? 1.f - __expf(-s1 * m.it1) : 0.f;
        const float q2 = s2 >= 0.f ? 1.f - __expf(-s2 * m.it2) : 0.f;
        const float r = x - fmaf(m.a, q2 - q1, m.i0);
        if (t < b1) r0 = fmaf(r, r, r0); else if (t < b2) r1 = fmaf(r, r, r1); else r2 = fmaf(r, r, r2);
    }
    double d0 = r0, d1 = r1, d2 = r2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        d0 += __shfl_xor_sync(CT_FULL, d0, o); d1 += __shfl_xor_sync(CT_FULL, d1, o); d2 += __shfl_xor_sync(CT_FULL, d2, o);
    }
    for (int i = lane; i <= a.max_levels; i += 32) ed[i] = -1;
    __syncwarp();
    if (lane == 0) {
        CT_CHECK_RANGE(ev * (a.max_levels + 1), 4, a.cap * (a.max_levels + 1), "stepfit, edge row");
        CT_CHECK_RANGE(ev * a.max_levels, 3, a.cap * a.max_levels, "stepfit, level row");
        ed[0] = 0; ed[1] = b1; ed[2] = b2; ed[3] = n;
        const double i0 = p[0] + (double)x0;
        double* mu_ = a.mean + ev * a.max_levels;
        double* sd_ = a.sd + ev * a.max_levels;
        mu_[0] = i0; mu_[1] = i0 - p[1]; mu_[2] = i0;
        sd_[0] = sqrt(d0 / b1); sd_[1] = sqrt(d1 / (b2 - b1)); sd_[2] = sqrt(d2 / (n - b2));
        a.n_levels[ev] = 3;
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

extern "C" int ct_stepfit_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end, int32_t* type,
                                const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0, int max_iters,
                                int max_levels, double* params6, double* cost, int32_t* iters, int32_t* n_levels, int32_t* edges,
                                double* level_mean, double* level_std, void* stream) {
    if (!y || !win_start || !win_end || !type || !params6 || !cost || !iters || !n_levels || !edges || !level_mean || !level_std) {
        ct_set_error("stepfit: null pointer"); return CT_ERR_ARG;
    }
    if (capacity < 0 || padding < 1 || padding > CT_STEPFIT_MAX_WINDOW || !(tau0 > 0.f) || max_iters < 1 || max_levels < 3) {
        ct_set_error("stepfit: bad argument (need padding >= 1, tau0 > 0, max_iters >= 1, max_levels >= 3)"); return CT_ERR_ARG;
    }
    if (capacity == 0) return CT_OK;
    if (capacity > 0x7fffffffLL * kSfWarps) { ct_set_error("stepfit: too many events in one batch"); return CT_ERR_UNSUPPORTED; }
    const int smem = kSfWarps * (int)sizeof(WarpSmem);
    if (cudaFuncSetAttribute(ct_stepfit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
        ct_set_error("stepfit: cannot reserve %d bytes of shared memory", smem); return CT_ERR_CUDA;
    }
    StepArgs a;
    a.y = y; a.ntot = n_total; a.w0 = (const long long*)win_start; a.w1 = (const long long*)win_end; a.type = type;
    a.nev_dev = (const long long*)n_events_dev; a.cap = capacity; a.padding = (int)padding; a.tau0 = tau0;
    a.max_iters = max_iters; a.max_levels = max_levels; a.params = params6; a.cost = cost; a.iters = iters;
    a.n_levels = n_levels; a.edges = edges; a.mean = level_mean; a.sd = level_std;
    const long long grid = (capacity + kSfWarps - 1) / kSfWarps;
    CT_COUNT_LAUNCH();
    ct_stepfit_kernel<<<(unsigned)grid, kSfWarps * 32, smem, (cudaStream_t)stream>>>(a);
    return ct_check_launch("ct_stepfit_kernel");
}
