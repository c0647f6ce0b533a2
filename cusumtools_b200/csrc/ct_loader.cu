// Loader-side device kernels: the byte formats either side of the hot path.
//   ct_bin_be_f64_to_f32 : ".bin" records (>f8 curr_pA, >f8 volt_mV) -> float32 pA
//                          (print_trace.py:33-34, noise-fit.py:90-91)
//   ct_i2be_to_f32       : legacy records (>i2 current, >i2 voltage) * savegain
//                          (legacy/minimal_psd.py:188-193)
//   ct_dequant_u16       : plot-trace.py:272-287 alone, for file series whose pieces have
//                          different gains (plot-trace.py:252-269) -> float32 path
//   ct_radix_hist_f32    : one digit pass of an exact radix select (np.pad(mode='median')
//                          for float input, plot-trace.py:319 applied to .bin data)
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {

__global__ void bin_be_kernel(const uint4* __restrict__ rec, long long n, float* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long st = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += st) {
        uint4 r = ct_ldg_stream(rec + i);                 // bytes 0-7: big-endian float64 current
        unsigned hi = __byte_perm(r.x, 0, 0x0123);        // most significant word, byte-swapped
        unsigned lo = __byte_perm(r.y, 0, 0x0123);
        out[i] = (float)__hiloint2double((int)hi, (int)lo);
    }
}
// savegain * current is a float64 product in the reference: rounded once to float32 here, not through a float32 gain
__global__ void i2be_kernel(const unsigned* __restrict__ rec, long long n, double gain, float* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long st = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += st) {
        unsigned r = rec[i];                              // bytes 0-1: big-endian int16 current
        short v = (short)(((r & 0xffu) << 8) | ((r >> 8) & 0xffu));
        out[i] = (float)(gain * (double)v);
    }
}
__global__ void dequant_kernel(const uint16_t* __restrict__ raw, long long n, unsigned mask, double alpha,
                               double beta, float* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long st = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += st) out[i] = (float)(alpha * (double)(raw[i] & mask) + beta);
}
__device__ __forceinline__ unsigned fkey(float v) {      // order-preserving float -> uint32
    unsigned b = __float_as_uint(v);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__global__ void __launch_bounds__(256)
radix_hist_kernel(const float* __restrict__ x, long long n, unsigned prefix, int prefix_bits, int use_abs,
                  unsigned long long* __restrict__ hist) {
    __shared__ unsigned sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const int shift = 32 - prefix_bits - 8;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long st = (long long)gridDim.x * blockDim.x;
    const long long nround = (n + st - 1) / st;
    for (long long r = 0; r < nround; ++r, i += st) {
        bool ok = i < n;
        unsigned k = 0;
        if (ok) {
            float v = x[i];
            k = fkey(use_abs ? fabsf(v) : v);
            ok = prefix_bits == 0 || (k >> (32 - prefix_bits)) == prefix;
        }
        const unsigned d = (k >> shift) & 0xffu;
        // warp-aggregated atomics: one shared-memory add per distinct digit per warp
        const unsigned act = __ballot_sync(CT_FULL, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(act, d);
            if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&sh[d], (unsigned)__popc(peers));
        }
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}

long long grid_for(long long n, int threads) {
    long long b = (n + threads - 1) / threads, cap = (long long)ct_sm_count() * 16;
    return b < 1 ? 1 : (b > cap ? cap : b);
}

}  // namespace

extern "C" {

int ct_bin_be_f64_to_f32(const void* records, int64_t n, float* out, void* stream) {
    if (!records || !out || n < 0 || (reinterpret_cast<uintptr_t>(records) & 15)) { ct_set_error("bin: bad argument / unaligned"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    CT_COUNT_LAUNCH();
    bin_be_kernel<<<(unsigned)grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)records, n, out);
    return ct_check_launch("bin_be_kernel");
}
int ct_i2be_to_f32(const void* records, int64_t n, double gain, float* out, void* stream) {
    if (!records || !out || n < 0 || (reinterpret_cast<uintptr_t>(records) & 3)) { ct_set_error("i2: bad argument / unaligned"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    CT_COUNT_LAUNCH();
    i2be_kernel<<<(unsigned)grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const unsigned*)records, n, gain, out);
    return ct_check_launch("i2be_kernel");
}
int ct_dequant_u16(const uint16_t* raw, int64_t n, uint16_t mask, double alpha, double beta, float* out, void* stream) {
    if (!raw || !out || n < 0) { ct_set_error("dequant: bad argument"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    CT_COUNT_LAUNCH();
    dequant_kernel<<<(unsigned)grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(raw, n, mask, alpha, beta, out);
    return ct_check_launch("dequant_kernel");
}
int ct_radix_hist_f32(const float* x, int64_t n, uint32_t prefix, int32_t prefix_bits, int32_t use_abs,
                      uint64_t* hist256, void* stream) {
    if (!x || !hist256 || n < 0 || prefix_bits < 0 || prefix_bits > 24 || prefix_bits % 8) { ct_set_error("radix_hist: bad argument"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    CT_COUNT_LAUNCH();
    radix_hist_kernel<<<(unsigned)grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, n, prefix, prefix_bits, use_abs, (unsigned long long*)hist256);
    return ct_check_launch("radix_hist_kernel");
}

}  // extern "C"
