// Zero-phase Bessel (plot-trace.py:313-320: filtfilt(b, a, np.pad(data, 1000, 'median'), padtype=None)) as
// two LANE-SEQUENTIAL passes for sm_100a, staged with TMA.
//
// Every lane owns whole RUNS of R consecutive samples and simply executes the recurrence (the reference's
// own dataflow, scipy _linear_filter, in cascade form): 4 FMA per section and sample.  A run starts Hw
// samples early (IIR warm-up, |h| tail < eps).  A warp owns 64 adjacent runs: lane l executes run l in the
// .x halves and run 32+l in the .y halves of float2 registers (FFMA2: two recurrences per issue slot, the
// only way to the 128 FMA/clk/SM of the B200).
//
// What decides the speed is the transposition between "lane = run" and "lane = consecutive address":
//   * forward INPUT (natural layout): one TMA 2-D tile copy per stage (cp.async.bulk.tensor.2d, box =
//     64 rows (runs, row stride R) x 128 bytes, SWIZZLE_128B, completion on an mbarrier), two stages per
//     warp; a lane then reads its own row with conflict-free LDS.128.  No per-lane copy instructions, no
//     address arithmetic, 16 KB of shared memory per warp (14 warps per SM).
//   * the SCRATCH between the passes is ours: it is kept lane-interleaved (unit = two 8-sample slots of the
//     32 lanes of one half-warp group, contiguous) so both passes move it with coalesced 128/256-bit accesses
//     straight from / into registers.  The forward output is band-limited by the filter itself, so only every
//     D-th sample is kept (D = 1, 2, 4, chosen on the host from the cascade's frequency response: the aliasing
//     error of "decimate, zero-stuff, filter backward" is max_f |H(f)| |H(f - k fs/D)|, required < 1e-7) and
//     the backward pass zero-stuffs it; the gain D rides on the forward pass's last section.
//   * final OUTPUT (natural layout): lanes write their rows into a swizzled half-tile (64 rows x 128 bytes)
//     and one TMA tile store per half-tile sends it out; dequantisation (offset + alpha*y) is folded into the
//     last section of the backward cascade (no extra instruction per sample).
// Groups of 64 runs that touch the ends of the trace (the median pad, partial tiles) take an EDGE
// instantiation with all the guards; everything else runs guard-free, straight-line code.
//
// Section arithmetic:  v[n] = x[n] + na1 v[n-1] + na2 v[n-2]        (all-pole part)
//                      y[n] = x[n] + (na1+n1) v[n-1] + (na2+n2) v[n-2]   (= v + n1 v1 + n2 v2)
// so the section output does not wait for v[n]: the cascade's dependent chain is 2 FMA per section.
//
// On its way out the backward pass can also (a) tally the baseline block sums of the final samples
// (ct_block_stats_f32 semantics, exact integers) and (b) leave the minimum / maximum of every 64-sample
// chunk, from which the detector classifies whole chunks without re-reading the trace (ct_detect.cu).
#include "ct_common.cuh"
#include "cusumtools_b200.h"
#include <cuda.h>
#include <math.h>
#include <string.h>
#include <stdlib.h>

namespace {

constexpr int kK = 64;              // samples per run per tile
constexpr int kG = 8;               // 8-sample slots per tile
constexpr int kRuns = 64;           // runs per warp (32 lanes x 2 halves)
constexpr int kStage = 8192;        // bytes per shared-memory stage / output half-tile: 64 rows x 128 B
constexpr int kWarps = 4;           // warps per CTA, one per SM sub-partition; 3 CTAs per SM (16 KB of shared memory per warp)
constexpr int kPfDist = 4;          // backward pass: scratch units are prefetched into L2 this many slot pairs ahead
constexpr int kCtasPerSm = 3;       // 12 warps per SM: three per scheduler, up to 168 registers each

typedef float2 f2;
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 splat(float v) { return make_float2(v, v); }

struct SeqArgs {
    const void* in;        // FWD: codes (uint16) or samples (float), natural layout; BWD: scratch
    float* out;            // scratch (FWD) or the final output, natural layout
    float2* summ;          // BWD, optional: (min, max) of every 64-sample chunk of the output, chunk c = positions base + 64c ..
    long long n_in;        // valid input positions [0, n_in): FWD n, BWD n + pad
    long long n_out;       // final output positions [0, n_out)
    long long ngroups;     // groups [g_first, ngroups) are processed
    long long g_first;
    long long scratch_runs;// runs the scratch holds
    long long scratch_floats, summ_count;   // extents of the scratch (floats) and of the chunk-extrema array (float2), for CT_BOUNDS_CHECK
    long long base;        // position of run 0 (<= 0): aligns groups with baseline blocks
    unsigned long long* next_group;   // work counter (zeroed by the host): warps fetch groups g_first + counter++ (NULL: static round robin)
    int R, Hw;             // run length, warm-up (multiples of kK, Hw <= R)
    int isub; unsigned mask; float fsub;   // uint16: x' = (code & mask) - isub; float: x' = x - fsub
    float pad_x;           // FWD: x' in the pad and beyond
    const float* pad_x_dev;// FWD, optional: added to pad_x on the device (the exact median arrives without a host round trip); 0 there: nothing to do
    float scale, offset;   // gain / offset folded into the last section (FWD scratch: D, 0)
    int tma_in, tma_out;   // tensor maps usable (alignment)
    // optional fused window count for the exact median (ct_count_window_u16 semantics), FWD uint16 only
    unsigned cw_k, cw_c; unsigned long long* cw_out; long long cw_p0, cw_p1;   // a = pat * cw_k + cw_c, see cw_tally2
    // optional fused baseline block statistics of the final output (ct_block_stats_f32 semantics)
    long long st_origin, st_block; float st_min, st_max, st_scale, st_nc0s;
    long long* st_cnt; long long* st_s1; long long* st_s2;
};

// ------------------------------------------------------------------ PTX helpers
static __device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
static __device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
static __device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
static __device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        :: "r"(bar), "r"(parity) : "memory");
}
static __device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap* map, int x, int y, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar) : "memory");
}
static __device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int x, int y, unsigned src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                 :: "l"(map), "r"(x), "r"(y), "r"(src) : "memory");
}
// the same with an L2 eviction policy (write-once output: evict_first keeps it from displacing lines that are still being filled)
static __device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* map, int x, int y, unsigned src, unsigned long long pol) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;"
                 :: "l"(map), "r"(x), "r"(y), "r"(src), "l"(pol) : "memory");
}
static __device__ __forceinline__ unsigned long long l2_stream_policy() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
static __device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> static __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory");
}
static __device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

static __device__ __forceinline__ uint4 lds128(unsigned addr) {
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
static __device__ __forceinline__ void sts128(unsigned addr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// swizzled (SWIZZLE_128B) byte offset of the 16-byte chunk c of row r inside a stage
static __device__ __forceinline__ unsigned swz(int r, int c) { return (unsigned)(r * 128 + ((c ^ (r & 7)) << 4)); }

template <int F> struct Vec { float v[F]; };
template <int F> static __device__ __forceinline__ void ldg_vec(const float* p, Vec<F>& r);
template <> __device__ __forceinline__ void ldg_vec<4>(const float* p, Vec<4>& r) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]) : "l"(p));
}
template <> __device__ __forceinline__ void ldg_vec<8>(const float* p, Vec<8>& r) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
}
template <> __device__ __forceinline__ void ldg_vec<16>(const float* p, Vec<16>& r) {
    Vec<8> a, b;
    ldg_vec<8>(p, a); ldg_vec<8>(p + 8, b);
#pragma unroll
    for (int i = 0; i < 8; ++i) { r.v[i] = a.v[i]; r.v[8 + i] = b.v[i]; }
}
template <int F> static __device__ __forceinline__ void stg_vec(float* p, const float* f);
template <> __device__ __forceinline__ void stg_vec<4>(float* p, const float* f) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" :: "l"(p), "f"(f[0]), "f"(f[1]), "f"(f[2]), "f"(f[3]) : "memory");
}
template <> __device__ __forceinline__ void stg_vec<8>(float* p, const float* f) {
    asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "f"(f[0]), "f"(f[1]), "f"(f[2]), "f"(f[3]), "f"(f[4]), "f"(f[5]), "f"(f[6]), "f"(f[7]) : "memory");
}
template <> __device__ __forceinline__ void stg_vec<16>(float* p, const float* f) { stg_vec<8>(p, f); stg_vec<8>(p + 8, f + 8); }
// 32-byte store that asks L2 to keep the line (evict_last): small pieces of the same line arrive tens of microseconds
// apart (chunk extrema: 32 bytes per run every four tiles) and should leave for DRAM as one line, not as four sectors.
static __device__ __forceinline__ unsigned long long l2_keep_policy() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
static __device__ __forceinline__ void stg8_keep(float* p, const float* f, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" :: "l"(p), "f"(f[0]), "f"(f[1]), "f"(f[2]), "f"(f[3]), "l"(pol) : "memory");
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" :: "l"(p + 4), "f"(f[4]), "f"(f[5]), "f"(f[6]), "f"(f[7]), "l"(pol) : "memory");
}

// ------------------------------------------------------------------ scratch layout
// Unit = the kept samples of one PAIR of slots (16 positions) of one run: F = 16/D floats.  Units of the 32
// runs of a half-warp group are contiguous (lane-interleaved): float offset of (run, tile to, pair jp).
template <int D>
static __device__ __forceinline__ long long scratch_off(long long run, int to, int jp, int TO) {
    constexpr int F = 16 / D;
    const long long g = run >> 6;
    const int h = (int)(run >> 5) & 1, l = (int)run & 31;
    return ((((g * TO + to) * 4 + jp) * 2 + h) * 32 + l) * F;
}

// ------------------------------------------------------------------ the cascade
// H(z) = g (1 + z^-1)^N / prod_s (1 - na1_s z^-1 - na2_s z^-2).  The all-pole sections run at every sample (2 FMA per
// section and sample, the section output IS its state); the numerator is one binomial FIR with the gain folded in,
// evaluated only where its output is needed (forward pass: at the kept positions, 9 taps per D samples) or only over
// the taps that see a non-zero input (backward pass: the zero-stuffed scratch, again 9 taps per D samples).  For the
// quarter-rate scratch that is 10.25 instead of 16 FMA per sample and pass - and, with the zeros at Nyquist applied
// last / first, 4x less rounding noise than the section-by-section form (0.005 pA against the float64 reference).
template <int NSEC> struct Coefs { f2 na1[NSEC], na2[NSEC], cf[2 * NSEC + 1], off; };
template <int NSEC>
__device__ __forceinline__ void load_coef(const CtFilterCoef& k, float out_gain, float offset, Coefs<NSEC>& c) {
#pragma unroll
    for (int s = 0; s < NSEC; ++s) { c.na1[s] = splat(k.na1[s]); c.na2[s] = splat(k.na2[s]); }
#pragma unroll
    for (int i = 0; i <= 2 * NSEC; ++i) c.cf[i] = splat(k.fir[i] * out_gain);
    c.off = splat(offset);
}
template <int NSEC>
__device__ __forceinline__ f2 allpole_step(f2 u, f2 (&v1)[NSEC], f2 (&v2)[NSEC], const Coefs<NSEC>& c) {
#pragma unroll
    for (int s = 0; s < NSEC; ++s) {
        const f2 vn = fma2(c.na1[s], v1[s], fma2(c.na2[s], v2[s], u));
        v2[s] = v1[s]; v1[s] = vn;
        u = vn;
    }
    return u;
}

// ------------------------------------------------------------------ exact-median window count (optional, FWD)
// counts[0] = #codes < lo, counts[1 + i] = #codes == lo + i*step for i < 8 (ct_count_window_u16 semantics), tallied from
// the float bit patterns the conversion has produced anyway: pat = 0x4B000000 + code, so a = pat*k + c with k = 4 / step and
// c = -(0x4B000000 + lo) k (mod 2^32) is 4 (code - lo) / step: its sign bit is the "below" count and 1 << a (PTX shl.b32
// CLAMPS amounts >= 32: nothing for codes above the window or below it) the increment of EIGHT 4-bit counters in one
// register.  After 8 tallies (a field holds at most 8) the even and the odd fields are added to two registers of 8-bit
// counters (5 instructions), which are emptied every 15 slots.  4.1 instructions per code (IMAD, LEA.HI, SHF.L, half an
// IADD3, 5/8 for the spreading): the pass is issue-bound once the tally rides on it, so every instruction per code costs
// 0.1 ms per 2.5 G samples (round-2 form: 8.5 per code).
static __device__ __forceinline__ unsigned shl_clamp(unsigned v, unsigned amt) {
    unsigned r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(amt));
    return r;
}
#ifndef CT_FWD_UNROLL
#define CT_FWD_UNROLL 1
#endif
// slots of the forward pass unrolled together: 1.98 ms with the tally at 1, 2.16 at 2, 2.38 at 4 (C2; without the tally
// 1.53 / 1.54 / 1.65): the loop body with the tally is 235 instructions, and the instruction cache decides
constexpr int kFwdUnroll = CT_FWD_UNROLL;
struct CwAcc { unsigned tot[9], below, c4, ce, co; int since; };
static __device__ __forceinline__ unsigned cw_amount(unsigned pat, const SeqArgs& a, unsigned cw_c) { return pat * a.cw_k + cw_c; }
static __device__ __forceinline__ void cw_tally2(unsigned pat0, unsigned pat1, const SeqArgs& a, unsigned cw_c, CwAcc& w) {
    const unsigned a0 = cw_amount(pat0, a, cw_c), a1 = cw_amount(pat1, a, cw_c);
    w.below += a0 >> 31;
    w.below += a1 >> 31;
    w.c4 += shl_clamp(1u, a0) + shl_clamp(1u, a1);
}
static __device__ __forceinline__ void cw_tally1(unsigned pat, const SeqArgs& a, unsigned cw_c, CwAcc& w) {
    const unsigned a0 = cw_amount(pat, a, cw_c);
    w.below += a0 >> 31;
    w.c4 += shl_clamp(1u, a0);
}
static __device__ __forceinline__ void cw_spread(CwAcc& w) {      // at most 8 tallies since the last call
    w.ce += w.c4 & 0x0f0f0f0fu;
    w.co += (w.c4 >> 4) & 0x0f0f0f0fu;
    w.c4 = 0;
}
static __device__ __forceinline__ void cw_flush(CwAcc& w) {       // at most 30 spreads since the last call
    w.tot[0] += w.below; w.below = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) { w.tot[1 + 2 * i] += (w.ce >> (8 * i)) & 0xffu; w.tot[2 + 2 * i] += (w.co >> (8 * i)) & 0xffu; }
    w.ce = 0; w.co = 0; w.since = 0;
}

// ------------------------------------------------------------------ output half-tiles (shared by FWD-final and BWD)
// Row r (0..63) of half-tile hb holds 32 consecutive floats of run run0 + r.  A lane writes the 8 samples of slot s
// (0..7 of the tile) of its two runs; after 4 slots the half-tile leaves through one TMA store (interior) or guarded
// scalar stores (trace edges / unaligned output).
static __device__ __forceinline__ void out_write_slot(unsigned outb, int lane, int s, const f2 (&y)[8]) {
    const unsigned hb = (unsigned)(s >> 2) * kStage;
    const int c = (s & 3) * 2;
    const unsigned a0 = outb + hb + swz(lane, c), a1 = outb + hb + swz(lane, c + 1);
    sts128(a0, y[0].x, y[1].x, y[2].x, y[3].x);
    sts128(a1, y[4].x, y[5].x, y[6].x, y[7].x);
    sts128(a0 + 32 * 128, y[0].y, y[1].y, y[2].y, y[3].y);
    sts128(a1 + 32 * 128, y[4].y, y[5].y, y[6].y, y[7].y);
}
// guarded copy of half-tile hb (positions first + r*R + [0, 32), r = 0..63) to the natural-layout output; the caller
// syncs the warp after it
static __device__ void out_store_guarded(const SeqArgs& a, unsigned outb, int hb, long long first, int lane) {
    for (int r = 0; r < kRuns; ++r) {
        const long long p = first + (long long)r * a.R + lane;
        float v;
        const unsigned addr = outb + (unsigned)hb * kStage + swz(r, lane >> 2) + (lane & 3) * 4;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
        if (p >= 0 && p < a.n_out) a.out[p] = v;
    }
    // this half-tile commits no bulk group, so the callers' paced waits (which count groups) would not cover a tile
    // store of the OTHER half that is still reading it when that half is rewritten next: drain them here
    if (lane == 0) bulk_wait_read<0>();
}

// ------------------------------------------------------------------ baseline block sums + chunk extrema (BWD epilogue)
// oracle/events_oracle.py::block_stats: q = rint((v - c0) 2^s) summed over the samples whose whole aligned 64-sample
// chunk lies inside [st_min, st_max].  A chunk is one tile row of a run, so a lane tallies its own chunks: the sums of
// the chunk in 32/64-bit partials, its extrema on the side (they are also what the detector wants), one verdict per
// chunk - no per-sample compare or select.
struct StatAcc { int c; long long s1, s2; };
struct ChunkAcc { int s1a, s1b; long long s2a, s2b; };      // chunk partials of the two halves
static __device__ __forceinline__ void tally_slot(const SeqArgs& a, ChunkAcc& k, const f2 (&y)[8]) {
    const f2 sc = splat(a.st_scale), nc = splat(a.st_nc0s);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        // (v - c0) * 2^s in one FFMA: scaling by a power of two commutes with the rounding of the difference
        const f2 t = fma2(y[e], sc, nc);
        const int u0 = __float2int_rn(t.x), u1 = __float2int_rn(t.y);
        k.s1a += u0; k.s1b += u1;
        k.s2a += (long long)u0 * u0; k.s2b += (long long)u1 * u1;
    }
}
// trace ends: sample by sample, only positions inside [0, n_out)
static __device__ __forceinline__ void tally_one(const SeqArgs& a, int& s1, long long& s2, float v) {
    const int q = __float2int_rn(__fmaf_rn(v, a.st_scale, a.st_nc0s));
    s1 += q; s2 += (long long)q * q;
}

static __device__ __forceinline__ float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }
static __device__ __forceinline__ float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// Work distribution: groups are handed out from a global counter (a warp that shares its scheduler with
// fewer or faster neighbours simply takes more of them; neighbouring groups are in flight together, which keeps
// their DRAM pages and L2 lines warm), or by static round robin when the caller gave no counter.
static __device__ __forceinline__ long long next_group(const SeqArgs& a, long long static_next, int lane, bool first) {
    if (!a.next_group) return first ? a.g_first + static_next : static_next;
    unsigned long long v = 0;
    if (lane == 0) v = atomicAdd(a.next_group, 1ULL);
    const long long i = (long long)__shfl_sync(CT_FULL, v, 0), span = a.ngroups - a.g_first;
    if (i >= span) return a.ngroups;
    // the last two groups (the right end of the trace: guarded, slow EDGE code) go out FIRST so that they run beside
    // the bulk of the work instead of after it; everything else in ascending order
    const long long ne = span < 2 ? span : 2;
    return i < ne ? a.ngroups - 1 - i : a.g_first + (i - ne);
}

// =============================== forward pass ========================================
// MODE: 1, 2, 4 = scratch output keeping every MODE-th sample; 0 = final output (causal filter only).
template <int NSEC, typename InT, int MODE, bool COUNT, bool EDGE>
__device__ __forceinline__ void fwd_group(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap* in_map, const CUtensorMap* out_map,
                                          const long long g, const int lane, const unsigned stage0, const unsigned bar0,
                                          const unsigned outb, unsigned& phase, const Coefs<NSEC>& cf, const float pad_x,
                                          const int isub, const unsigned cw_c) {
    constexpr bool U16 = sizeof(InT) == 2;
    constexpr int SPT = U16 ? 1 : 2;             // stages per tile (a stage row is 128 bytes)
    constexpr int SLOTS = kG / SPT;              // slots per stage
    constexpr int SAMP = kK / SPT;               // samples per stage row
    constexpr int D = MODE ? MODE : 1;
    constexpr int F = 16 / D;
    const long long run0 = g * kRuns;
    const int ntiles = (a.Hw + a.R) / kK, wt = a.Hw / kK, TO = a.R / kK;
    const int nstages = ntiles * SPT;
    const InT* in = reinterpret_cast<const InT*>(a.in);
    const unsigned m2 = a.mask | (a.mask << 16);
    const f2 kmagic = splat(-(8388608.f + (float)isub));

    constexpr int TAPS = 2 * NSEC + 1;              // binomial FIR taps (orders below 2 NSEC have zero tails)
    constexpr int HIST = TAPS - 1 > 8 ? 16 : 8;     // all-pole outputs of the previous slot(s) the FIR reaches back into
    f2 v1[NSEC], v2[NSEC], ahist[HIST];
    {   // runs that begin in the left pad start from the steady state of the pad value (scipy: zi * x[0])
        float p0 = 0.f, p1 = 0.f;
        if (EDGE) {
            p0 = a.base + (run0 + lane) * a.R - a.Hw < 0 ? pad_x : 0.f;
            p1 = a.base + (run0 + lane + 32) * a.R - a.Hw < 0 ? pad_x : 0.f;
        }
#pragma unroll
        for (int s = 0; s < NSEC; ++s) { v1[s] = make_float2(p0 * k.ss[s], p1 * k.ss[s]); v2[s] = v1[s]; }
#pragma unroll
        for (int i = 0; i < HIST; ++i) ahist[i] = v1[NSEC - 1];
    }
    CwAcc cw;
    if (COUNT) {
#pragma unroll
        for (int i = 0; i < 9; ++i) cw.tot[i] = 0;
        cw.below = cw.c4 = cw.ce = cw.co = 0; cw.since = 0;
    }

    // stage q covers the positions base + (run0 + r) R + off(q) + [0, SAMP), r = 0..63
    auto stage_off = [&](int q) { return (long long)(q / SPT) * kK - a.Hw + (q % SPT) * SAMP; };
    auto issue = [&](int q) {
        const long long off = stage_off(q);
        const unsigned buf = stage0 + (unsigned)(q & 1) * kStage, bar = bar0 + (unsigned)(q & 1) * 8;
        bool tma = true;                             // interior groups: every stage is one tile copy
        if (EDGE) {
            const long long first = a.base + run0 * a.R + off;
            tma = a.tma_in && first >= 0 && first + (long long)(kRuns - 1) * a.R + SAMP <= a.n_in;
        }
        if (tma) {
            if (lane == 0) {
                mbar_expect_tx(bar, kStage);
                // warm-up pieces (off < 0) are the tail of the previous run: one row up, R further right
                const int x = off >= 0 ? (int)off : (int)(a.R + off);
                const int y = (int)(run0) - (off >= 0 ? 0 : 1);
                tma_load_2d(buf, in_map, x, y, bar);
            }
        } else if (EDGE) {
            // guarded fill of the same swizzled layout; float gets the pad value outside the data, codes are fixed up later
            constexpr int EPC = 16 / (int)sizeof(InT);      // elements per 16-byte chunk
            for (int r = 0; r < kRuns; ++r) {
#pragma unroll
                for (int half = 0; half < (SAMP > 32 ? 2 : 1); ++half) {
                    const int col = lane + half * 32;
                    const long long p = a.base + (run0 + r) * a.R + off + col;
                    InT v;
                    if (U16) v = (p >= 0 && p < a.n_in) ? in[p] : (InT)0;
                    else v = (p >= 0 && p < a.n_in) ? in[p] : (InT)(a.fsub + pad_x);
                    const unsigned addr = buf + swz(r, col / EPC) + (unsigned)(col % EPC) * (unsigned)sizeof(InT);
                    if (U16) asm volatile("st.shared.u16 [%0], %1;" :: "r"(addr), "h"((unsigned short)v) : "memory");
                    else asm volatile("st.shared.f32 [%0], %1;" :: "r"(addr), "f"((float)v) : "memory");
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar);
        }
    };

    issue(0);
    f2 keep[F];                                     // kept samples of the current slot pair (scratch modes)
    for (int t = 0; t < ntiles; ++t) {
        const bool store = t >= wt;
        const long long toff = (long long)t * kK - a.Hw;
        const long long lo0 = a.base + (run0 + lane) * a.R + toff, lo1 = lo0 + 32LL * a.R;
        const bool edge = EDGE && U16 && !(lo0 >= 0 && lo1 + kK <= a.n_in);
        const bool cw_part = COUNT && EDGE && !(lo0 >= a.cw_p0 && lo1 + kK <= a.cw_p1 && lo0 + kK <= a.cw_p1 && lo1 >= a.cw_p0);
#pragma unroll
        for (int hs = 0; hs < SPT; ++hs) {
            const int q = t * SPT + hs;
            if (q + 1 < nstages) issue(q + 1);
            const unsigned buf = stage0 + (unsigned)(q & 1) * kStage;
            mbar_wait(bar0 + (unsigned)(q & 1) * 8, (phase >> (q & 1)) & 1u);
            phase ^= 1u << (q & 1);
            const unsigned row0 = buf + (unsigned)lane * 128u;
            const int sw = lane & 7;
            if (MODE == 0 && store && hs == 0 && a.tma_out) {   // the half-tile about to be rewritten must have left
                if (lane == 0) bulk_wait_read<1>();
                __syncwarp();
            }
#pragma unroll kFwdUnroll
            for (int j = 0; j < SLOTS; ++j) {
                const int jj = hs * SLOTS + j;             // slot inside the tile
                f2 x[8];
                if (U16) {
                    const uint4 ra = lds128(row0 + (unsigned)((j ^ sw) << 4));
                    const uint4 rb = lds128(row0 + 32 * 128 + (unsigned)((j ^ sw) << 4));
                    const unsigned wa[4] = {ra.x & m2, ra.y & m2, ra.z & m2, ra.w & m2};
                    const unsigned wb[4] = {rb.x & m2, rb.y & m2, rb.z & m2, rb.w & m2};
                    unsigned pl[4][2], ph[4][2];           // 2^23 + code as float bit patterns (byte permute): [word][run]
#pragma unroll
                    for (int w = 0; w < 4; ++w) {
                        pl[w][0] = __byte_perm(wa[w], 0x4B000000u, 0x7410); pl[w][1] = __byte_perm(wb[w], 0x4B000000u, 0x7410);
                        ph[w][0] = __byte_perm(wa[w], 0x4B000000u, 0x7432); ph[w][1] = __byte_perm(wb[w], 0x4B000000u, 0x7432);
                        // minus (2^23 + isub): exact
                        x[2 * w] = __fadd2_rn(make_float2(__uint_as_float(pl[w][0]), __uint_as_float(pl[w][1])), kmagic);
                        x[2 * w + 1] = __fadd2_rn(make_float2(__uint_as_float(ph[w][0]), __uint_as_float(ph[w][1])), kmagic);
                    }
                    if (edge) {                            // x' = pad_x in the pad and beyond it
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const long long p0 = lo0 + jj * 8 + e, p1 = lo1 + jj * 8 + e;
                            if (!(p0 >= 0 && p0 < a.n_in)) x[e].x = pad_x;
                            if (!(p1 >= 0 && p1 < a.n_in)) x[e].y = pad_x;
                        }
                    }
                    if (COUNT && store) {                  // every code of [cw_p0, cw_p1) is tallied exactly once
                        if (!cw_part) {
#pragma unroll
                            for (int w = 0; w < 4; ++w) {
                                cw_tally2(pl[w][0], ph[w][0], a, cw_c, cw);
                                cw_tally2(pl[w][1], ph[w][1], a, cw_c, cw);
                                if (w & 1) cw_spread(cw);      // 8 tallies
                            }
                        } else {
#pragma unroll 1
                            for (int w = 0; w < 4; ++w) {
                                const long long pa0 = lo0 + jj * 8 + 2 * w, pb0 = lo1 + jj * 8 + 2 * w;
                                if (pa0 >= a.cw_p0 && pa0 < a.cw_p1) cw_tally1(pl[w][0], a, cw_c, cw);
                                if (pa0 + 1 >= a.cw_p0 && pa0 + 1 < a.cw_p1) cw_tally1(ph[w][0], a, cw_c, cw);
                                if (pb0 >= a.cw_p0 && pb0 < a.cw_p1) cw_tally1(pl[w][1], a, cw_c, cw);
                                if (pb0 + 1 >= a.cw_p0 && pb0 + 1 < a.cw_p1) cw_tally1(ph[w][1], a, cw_c, cw);
                                if (w & 1) cw_spread(cw);
                            }
                        }
                        if (++cw.since == 15) cw_flush(cw);   // two spreads of <= 8 per slot: an 8-bit counter holds 15 slots
                    }
                } else {
                    const uint4 a0 = lds128(row0 + (unsigned)(((2 * j) ^ sw) << 4)), a1 = lds128(row0 + (unsigned)(((2 * j + 1) ^ sw) << 4));
                    const uint4 b0 = lds128(row0 + 32 * 128 + (unsigned)(((2 * j) ^ sw) << 4));
                    const uint4 b1 = lds128(row0 + 32 * 128 + (unsigned)(((2 * j + 1) ^ sw) << 4));
                    const unsigned wa[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                    const unsigned wb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                    const f2 nsub = splat(-a.fsub);
#pragma unroll
                    for (int e = 0; e < 8; ++e) x[e] = __fadd2_rn(make_float2(__uint_as_float(wa[e]), __uint_as_float(wb[e])), nsub);
                }
                f2 ap[8];                                  // all-pole output of the slot
#pragma unroll
                for (int e = 0; e < 8; ++e) ap[e] = allpole_step<NSEC>(x[e], v1, v2, cf);
                if (store) {
                    // numerator (+ gain, + offset in the final-output mode) at the positions that are kept
#pragma unroll
                    for (int e = 0; e < 8; e += D) {
                        f2 y = MODE == 0 ? fma2(cf.cf[0], ap[e], cf.off) : __fmul2_rn(cf.cf[0], ap[e]);
#pragma unroll
                        for (int t2 = 1; t2 < TAPS; ++t2) y = fma2(cf.cf[t2], e - t2 >= 0 ? ap[e - t2 >= 0 ? e - t2 : 0] : ahist[HIST + e - t2], y);
                        x[e] = y;
                    }
                }
                if (HIST == 16) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) ahist[i] = ahist[8 + i];
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) ahist[HIST - 8 + i] = ap[i];
                if (store) {
                    if (MODE == 0) {
                        out_write_slot(outb, lane, jj, x);
                        if ((jj & 3) == 3) {               // half-tile complete
                            const int hb = jj >> 2;
                            const long long first = a.base + run0 * a.R + toff + hb * 32;
                            bool tma = true;
                            if (EDGE) tma = a.tma_out && first >= 0 && first + (long long)(kRuns - 1) * a.R + 32 <= a.n_out;
                            if (tma) {
                                fence_async_smem();
                                __syncwarp();
                                if (lane == 0) {
                                    tma_store_2d(out_map, (int)(toff + hb * 32), (int)run0, outb + (unsigned)hb * kStage);
                                    bulk_commit();
                                }
                                if (hb == 0) {             // the other half is rewritten next
                                    if (lane == 0) bulk_wait_read<1>();
                                    __syncwarp();
                                }
                            } else if (EDGE) {
                                __syncwarp();
                                out_store_guarded(a, outb, hb, first, lane);
                                __syncwarp();
                            }
                        }
                    } else {
                        // keep every D-th sample; a pair of slots fills one scratch unit of F floats per half
                        constexpr int PER = 8 / D;
#pragma unroll
                        for (int i = 0; i < PER; ++i) keep[(jj & 1) * PER + i] = x[i * D];
                        if (jj & 1) {
                            float oa[F], ob[F];
#pragma unroll
                            for (int i = 0; i < F; ++i) { oa[i] = keep[i].x; ob[i] = keep[i].y; }
                            const long long so = scratch_off<D>(run0 + lane, t - wt, jj >> 1, TO);
                            CT_CHECK_RANGE(so, 33 * F, a.scratch_floats, "forward pass, scratch store");
                            float* dst = a.out + so;
                            stg_vec<F>(dst, oa);
                            stg_vec<F>(dst + 32 * F, ob);
                        }
                    }
                }
            }
            __syncwarp();                                  // every lane is done with the stage before it is refilled
        }
    }
    if (COUNT) {                                           // (a lane tallies < 2^32 codes per group)
        cw_flush(cw);
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            unsigned v = cw.tot[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CT_FULL, v, o);
            if (lane == 0 && v) atomicAdd(a.cw_out + i, (unsigned long long)v);
        }
    }
}

template <int NSEC, typename InT, int MODE, bool COUNT>
__global__ void __launch_bounds__(kWarps * 32, kCtasPerSm)
ct_filter_fwd_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ CUtensorMap out_map, SeqArgs a, CtFilterCoef k,
                     const CtMedianPlan* __restrict__ plan) {
    // plan (uint16, may be NULL): sub and the count window's first code come from the estimate on the device; isub = floor(sub),
    // cw_c from lo, and the fraction of sub joins pad_x, as split_sub and the host do for the values passed in `a`.  (Its own
    // argument: a field of SeqArgs would move the coefficients behind it off the alignment of their 128-bit constant loads.)
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int kPerWarp = 2 * kStage + (MODE == 0 ? 2 * kStage : 0);
    const int lane = ct_lane();
    const int wib = threadIdx.x >> 5;
    float pad_x = a.pad_x;
    int isub = a.isub;
    unsigned cw_c = a.cw_c;
    if (sizeof(InT) == 2 && plan) {
        const float sub = __ldg(&plan->sub_code), fl = floorf(sub);
        isub = (int)fl;
        pad_x += sub - fl;
        if (COUNT) cw_c = 0u - (0x4B000000u + __ldg(&plan->lo)) * a.cw_k;
    }
    if (a.pad_x_dev) {                                       // the end groups re-run with the exact median's pad: a no-op when
        const float d = __ldg(a.pad_x_dev);                  // the estimate was the median
        if (d == 0.f) return;
        pad_x += d;
    }
    const unsigned sbase = smem_u32(smem);
    const unsigned stage0 = sbase + (unsigned)wib * kPerWarp;
    const unsigned outb = stage0 + 2 * kStage;
    const unsigned bar0 = sbase + (unsigned)kWarps * kPerWarp + (unsigned)wib * 16;
    if (lane == 0) {
        if (sbase & 1023u) asm volatile("trap;");
        mbar_init(bar0, 1); mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    __syncwarp();
    const long long gw = (long long)blockIdx.x * kWarps + wib;
    const long long nw = (long long)gridDim.x * kWarps;

    Coefs<NSEC> cf;
    load_coef<NSEC>(k, a.scale, a.offset, cf);
    unsigned phase = 0;
    for (long long g = next_group(a, gw, lane, true); g < a.ngroups; g = next_group(a, g + nw, lane, false)) {
        // interior groups (every stage and output piece of all 64 runs inside the data, the counted range too) run guard-free
        const long long p_lo = a.base + g * kRuns * a.R - a.Hw, p_hi = a.base + (g + 1) * kRuns * a.R;
        bool interior = a.tma_in && p_lo >= 0 && p_hi <= a.n_in;
        if (MODE == 0) interior = interior && a.tma_out && p_hi <= a.n_out;
        if (COUNT) interior = interior && p_lo + a.Hw >= a.cw_p0 && p_hi <= a.cw_p1;
        if (interior) fwd_group<NSEC, InT, MODE, COUNT, false>(a, k, &in_map, &out_map, g, lane, stage0, bar0, outb, phase, cf, pad_x, isub, cw_c);
        else fwd_group<NSEC, InT, MODE, COUNT, true>(a, k, &in_map, &out_map, g, lane, stage0, bar0, outb, phase, cf, pad_x, isub, cw_c);
    }
    if (MODE == 0 && lane == 0) bulk_wait_read<0>();         // shared memory must outlive the last tile store
}

// =============================== backward pass =======================================
// Run r processes positions r*R + R + Hw - 1 down to r*R, the first Hw of them (the first Hw/K tiles of run
// r + 1) only to warm the recursion up.  The scratch holds D * (forward output) at every D-th position.
template <int NSEC, int D, bool STATS, bool SUMM, bool EDGE>
__device__ __forceinline__ void bwd_group(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap* out_map, const long long g,
                                          const int lane, const unsigned outb, const float hold_d, const Coefs<NSEC>& cf) {
    constexpr int F = 16 / D;
    const float* y1 = reinterpret_cast<const float*>(a.in);
    const long long run0 = g * kRuns;
    const long long r0 = run0 + lane, r1 = r0 + 32;
    const int ntiles = (a.Hw + a.R) / kK, wt = a.Hw / kK, TO = a.R / kK;
    const int npairs = ntiles * 4;

    constexpr int TAPS = 2 * NSEC + 1;              // binomial FIR taps
    constexpr int PER = 8 / D;                      // kept samples per slot
    constexpr int NW = (8 + TAPS - 1 + D - 1) / D;  // window of kept samples the FIR of one slot reaches: positions [0, 8 + TAPS - 1)
    f2 v1[NSEC], v2[NSEC], zw[NW];
    {   // Runs whose first processed position lies beyond the data start from the steady state of the held value
        // (scipy: zi * y[-1], _signaltools.py:4910-4913).  Beyond the data the scratch is the zero-stuffed constant
        // hold_d, whose mean is hold_d / D: the FIR's DC output times the all-pole steady-state factors.
        float h0 = 0.f, h1 = 0.f;
        if (EDGE) {
            h0 = a.base + r0 * a.R + a.R + a.Hw - 1 >= a.n_in ? hold_d : 0.f;
            h1 = a.base + r1 * a.R + a.R + a.Hw - 1 >= a.n_in ? hold_d : 0.f;
        }
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < TAPS; ++i) sum += cf.cf[i].x;
        const float w0 = h0 * sum * (1.f / (float)D), w1 = h1 * sum * (1.f / (float)D);
#pragma unroll
        for (int s = 0; s < NSEC; ++s) { v1[s] = make_float2(w0 * k.ss[s], w1 * k.ss[s]); v2[s] = v1[s]; }
#pragma unroll
        for (int i = 0; i < NW; ++i) zw[i] = make_float2(h0, h1);
    }
    // pair i (0 .. npairs-1) in processing order: tile t = i / 4, pair jp = 3 - i % 4 (descending positions)
    auto fetch = [&](int i, Vec<F>& xa, Vec<F>& xb) {
        const int t = i >> 2, jp = 3 - (i & 3);
        const bool warm = t < wt;
        const int to = warm ? wt - 1 - t : TO - 1 - (t - wt);
        const long long s0 = warm ? r0 + 1 : r0, s1 = warm ? r1 + 1 : r1;
        if (!EDGE) {
            CT_CHECK_RANGE(scratch_off<D>(s0, to, jp, TO), F, a.scratch_floats, "backward pass, scratch load (half 0)");
            CT_CHECK_RANGE(scratch_off<D>(s1, to, jp, TO), F, a.scratch_floats, "backward pass, scratch load (half 1)");
            ldg_vec<F>(y1 + scratch_off<D>(s0, to, jp, TO), xa);
            ldg_vec<F>(y1 + scratch_off<D>(s1, to, jp, TO), xb);
            // the register pipeline is two pairs deep (about a microsecond of work): it hides an L2 hit, not a DRAM
            // access under load, so the units of the pair kPfDist further on are pulled into L2 now (both halves of
            // a pair are contiguous: 256 F bytes, one line per lane)
            const int ip = i + kPfDist;
            if (ip < npairs && lane < 2 * F) {
                const int tp = ip >> 2, jpp = 3 - (ip & 3);
                const bool wp = tp < wt;
                const int top = wp ? wt - 1 - tp : TO - 1 - (tp - wt);
                const float* pf = y1 + scratch_off<D>(run0 + (wp ? 1 : 0), top, jpp, TO) + lane * 32;
                asm volatile("prefetch.global.L2 [%0];" :: "l"(pf));
            }
        } else {
            // units beyond the scratch are never dereferenced; positions beyond the forward output are replaced by `hold` below
            if (s0 < a.scratch_runs) { CT_CHECK_RANGE(scratch_off<D>(s0, to, jp, TO), F, a.scratch_floats, "backward pass (edge), scratch load"); ldg_vec<F>(y1 + scratch_off<D>(s0, to, jp, TO), xa); }
            if (s1 < a.scratch_runs) { CT_CHECK_RANGE(scratch_off<D>(s1, to, jp, TO), F, a.scratch_floats, "backward pass (edge), scratch load"); ldg_vec<F>(y1 + scratch_off<D>(s1, to, jp, TO), xb); }
        }
    };
    StatAcc acc0, acc1;
    acc0.c = 0; acc0.s1 = 0; acc0.s2 = 0; acc1 = acc0;
    float2 sb0[4], sb1[4];                          // chunk extrema of four consecutive tiles (one 32-byte store each)
    Vec<F> pa[2], pb[2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int e = 0; e < F; ++e) { pa[i].v[e] = 0.f; pb[i].v[e] = 0.f; }
    fetch(0, pa[0], pb[0]);
    if (npairs > 1) fetch(1, pa[1], pb[1]);

    for (int t = 0; t < ntiles; ++t) {
        const bool warm = t < wt;
        const bool store = !warm;
        const int to = warm ? wt - 1 - t : TO - 1 - (t - wt);
        const long long tpos0 = a.base + (warm ? r0 + 1 : r0) * a.R + (long long)to * kK;   // position of the tile's first sample, half 0
        float mn0 = __int_as_float(0x7f800000), mx0 = __int_as_float(0xff800000), mn1 = mn0, mx1 = mx0;
        ChunkAcc ck; ck.s1a = ck.s1b = 0; ck.s2a = ck.s2b = 0;     // the tile row of each run is one chunk of the in-window rule
        int have0 = EDGE ? 0 : kK, have1 = have0;                    // samples of the chunk that exist (trace ends)
#pragma unroll 1
        for (int jq = 0; jq < 4; ++jq) {
            const int jp = 3 - jq;
            // the unit of this pair -> x registers; shift the pipeline, issue the pair after next
            Vec<F> ca = pa[0], cb = pb[0];
            pa[0] = pa[1]; pb[0] = pb[1];
            { const int nx = t * 4 + jq + 2; if (nx < npairs) fetch(nx, pa[1], pb[1]); }
            if (!EDGE) {
                // interior groups send both half-tiles of a tile together (below): the tile's previous stores must have
                // read the buffers before its first slot is written
                if (store && jq == 0) {
                    if (lane == 0) bulk_wait_read<0>();
                    __syncwarp();
                }
            } else if (store && (jq & 1) == 0 && a.tma_out) {     // this half-tile's previous store must have read it
                if (lane == 0) bulk_wait_read<1>();
                __syncwarp();
            }
#pragma unroll
            for (int sl = 1; sl >= 0; --sl) {              // upper slot of the pair first (rolled: 2.66 ms against 2.44 ms)
                const int jj = jp * 2 + sl;
                // the slot's kept samples enter the window at positions 0, D, ..; the entries above came down from the
                // slots processed before (higher positions)
#pragma unroll
                for (int i = NW - 1; i >= PER; --i) zw[i] = zw[i - PER];
#pragma unroll
                for (int i = 0; i < PER; ++i) zw[i] = make_float2(ca.v[sl * PER + i], cb.v[sl * PER + i]);
                if (EDGE) {
                    const long long q0 = tpos0 + jj * 8, q1 = q0 + 32LL * a.R;
                    if (q1 + 8 > a.n_in) {                 // (q0 < q1) beyond the forward output: the held value
#pragma unroll
                        for (int i = 0; i < PER; ++i) {
                            if (q0 + i * D >= a.n_in) zw[i].x = hold_d;
                            if (q1 + i * D >= a.n_in) zw[i].y = hold_d;
                        }
                    }
                }
                f2 x[8];
#pragma unroll
                for (int ee = 0; ee < 8; ++ee) {
                    const int e = 7 - ee;
                    // numerator over the zero-stuffed scratch: only the taps that meet a kept position, e <= i D <= e + TAPS - 1
                    f2 w = make_float2(0.f, 0.f);
                    bool first = true;
#pragma unroll
                    for (int i = 0; i < NW; ++i) {
                        const int t2 = i * D - e;
                        if (t2 >= 0 && t2 < TAPS) { w = first ? __fmul2_rn(cf.cf[t2], zw[i]) : fma2(cf.cf[t2], zw[i], w); first = false; }
                    }
                    x[e] = __fadd2_rn(allpole_step<NSEC>(w, v1, v2, cf), cf.off);
                }
                if (store) {
                    out_write_slot(outb, lane, jj, x);
                    if (!EDGE) {
                        if (STATS) tally_slot(a, ck, x);
                        if (STATS || SUMM) {
#pragma unroll
                            for (int e = 0; e < 8; e += 2) {
                                mn0 = fmin3(mn0, x[e].x, x[e + 1].x); mx0 = fmax3(mx0, x[e].x, x[e + 1].x);
                                mn1 = fmin3(mn1, x[e].y, x[e + 1].y); mx1 = fmax3(mx1, x[e].y, x[e + 1].y);
                            }
                        }
                    } else {
                        const long long p0 = a.base + r0 * a.R + (long long)to * kK + jj * 8, p1 = p0 + 32LL * a.R;
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            if (p0 + e >= 0 && p0 + e < a.n_out) {
                                if (STATS) tally_one(a, ck.s1a, ck.s2a, x[e].x);
                                mn0 = fminf(mn0, x[e].x); mx0 = fmaxf(mx0, x[e].x); ++have0;
                            }
                            if (p1 + e >= 0 && p1 + e < a.n_out) {
                                if (STATS) tally_one(a, ck.s1b, ck.s2b, x[e].y);
                                mn1 = fminf(mn1, x[e].y); mx1 = fmaxf(mx1, x[e].y); ++have1;
                            }
                        }
                    }
                }
            }
            if (!EDGE) {
                // Both half-tiles leave at the end of the tile: the two 128-byte lines of a run's 256 bytes reach L2 (and
                // DRAM) together.  With 113 664 output streams in flight the write-back granularity decides the DRAM
                // efficiency (scripts/ubench/stride_bw.cu: 4.4 TB/s at 128 bytes at a time, 5.1 at 256 for this mix).
                if (store && jq == 3) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        const unsigned long long pol = l2_stream_policy();
                        tma_store_2d_hint(out_map, to * kK, (int)run0, outb, pol);
                        tma_store_2d_hint(out_map, to * kK + 32, (int)run0, outb + (unsigned)kStage, pol);
                        bulk_commit();
                    }
                }
            } else if (store && (jq & 1)) {                // half-tile hb = jp >> 1 complete
                const int hb = jp >> 1;
                const long long first = a.base + run0 * a.R + (long long)to * kK + hb * 32;
                bool tma = true;
                if (EDGE) tma = a.tma_out && first >= 0 && first + (long long)(kRuns - 1) * a.R + 32 <= a.n_out;
                if (tma) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_2d(out_map, to * kK + hb * 32, (int)run0, outb + (unsigned)hb * kStage);
                        bulk_commit();
                    }
                } else if (EDGE) {
                    __syncwarp();
                    out_store_guarded(a, outb, hb, first, lane);
                    __syncwarp();
                }
            }
        }
        if (STATS && store) {                              // the chunk's verdict: every existing sample inside the window
            if (have0 > 0 && mn0 >= a.st_min && mx0 <= a.st_max) { acc0.c += have0; acc0.s1 += ck.s1a; acc0.s2 += ck.s2a; }
            if (have1 > 0 && mn1 >= a.st_min && mx1 <= a.st_max) { acc1.c += have1; acc1.s1 += ck.s1b; acc1.s2 += ck.s2b; }
        }
        if (SUMM && store) {
            // tiles descend: the newest chunk is the lowest one of its group of four
            sb0[3] = sb0[2]; sb0[2] = sb0[1]; sb0[1] = sb0[0]; sb0[0] = make_float2(mn0, mx0);
            sb1[3] = sb1[2]; sb1[2] = sb1[1]; sb1[1] = sb1[0]; sb1[0] = make_float2(mn1, mx1);
            if ((to & 3) == 0) {
                CT_CHECK_RANGE(r0 * TO + to, 4, a.summ_count, "backward pass, chunk extrema (half 0)");
                CT_CHECK_RANGE(r1 * TO + to, 4, a.summ_count, "backward pass, chunk extrema (half 1)");
                float2* d0 = a.summ + (r0 * TO + to);
                float2* d1 = a.summ + (r1 * TO + to);
                const float f0[8] = {sb0[0].x, sb0[0].y, sb0[1].x, sb0[1].y, sb0[2].x, sb0[2].y, sb0[3].x, sb0[3].y};
                const float f1[8] = {sb1[0].x, sb1[0].y, sb1[1].x, sb1[1].y, sb1[2].x, sb1[2].y, sb1[3].x, sb1[3].y};
                const unsigned long long keep = l2_keep_policy();
                stg8_keep(reinterpret_cast<float*>(d0), f0, keep);
                stg8_keep(reinterpret_cast<float*>(d1), f1, keep);
            }
        }
    }
    if (STATS) {                                           // the group lies inside one baseline block (grid aligned by `base`)
        long long c = (long long)acc0.c + acc1.c, s1 = acc0.s1 + acc1.s1, s2 = acc0.s2 + acc1.s2;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c += __shfl_xor_sync(CT_FULL, c, o); s1 += __shfl_xor_sync(CT_FULL, s1, o); s2 += __shfl_xor_sync(CT_FULL, s2, o);
        }
        const long long rel = a.base + run0 * a.R - a.st_origin;
        if (lane == 0 && c && rel >= 0) {
            const long long kb = rel / a.st_block;
            atomicAdd(reinterpret_cast<unsigned long long*>(a.st_cnt + kb), (unsigned long long)c);
            atomicAdd(reinterpret_cast<unsigned long long*>(a.st_s1 + kb), (unsigned long long)s1);
            atomicAdd(reinterpret_cast<unsigned long long*>(a.st_s2 + kb), (unsigned long long)s2);
        }
    }
}

template <int NSEC, int D, bool STATS, bool SUMM>
__global__ void __launch_bounds__(kWarps * 32, kCtasPerSm)
ct_filter_bwd_kernel(const __grid_constant__ CUtensorMap out_map, SeqArgs a, CtFilterCoef k) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int lane = ct_lane();
    const int wib = threadIdx.x >> 5;
    const unsigned sbase = smem_u32(smem);
    const unsigned outb = sbase + (unsigned)wib * 2 * kStage;
    if (lane == 0 && (sbase & 1023u)) asm volatile("trap;");
    const float* y1 = reinterpret_cast<const float*>(a.in);
    const long long gw = (long long)blockIdx.x * kWarps + wib;
    const long long nw = (long long)gridDim.x * kWarps;
    const int TO = a.R / kK;

    Coefs<NSEC> cf;
    load_coef<NSEC>(k, a.scale, a.offset, cf);
    // the forward output is held constant beyond n_in (scipy: the backward pass starts from zi * y[-1]): as a scratch
    // entry, i.e. D times its last kept sample (the output is flat at the end of the pad)
    const long long last = (a.n_in - 1 - a.base) / D * D;                  // relative to the run grid
    const int lo = (int)(last % a.R);
    const float hold_d = y1[scratch_off<D>(last / a.R, lo / kK, (lo % kK) >> 4, TO) + (lo & 15) / D];

    for (long long g = next_group(a, gw, lane, true); g < a.ngroups; g = next_group(a, g + nw, lane, false)) {
        const long long p_lo = a.base + g * kRuns * a.R, p_hi = a.base + (g + 1) * kRuns * a.R;
        const bool interior = a.tma_out && p_lo >= 0 && p_hi + a.Hw <= a.n_in && p_hi <= a.n_out && (g + 1) * kRuns < a.scratch_runs;
        if (lane == 0) bulk_wait_read<0>();                // (the two group variants pace their tile stores differently)
        __syncwarp();
        if (interior) bwd_group<NSEC, D, STATS, SUMM, false>(a, k, &out_map, g, lane, outb, hold_d, cf);
        else bwd_group<NSEC, D, STATS, SUMM, true>(a, k, &out_map, g, lane, outb, hold_d, cf);
    }
    if (lane == 0) bulk_wait_read<0>();                    // shared memory must outlive the last tile store
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        cudaGetLastError();
    }
    return fn;
}
// 2-D view of a trace as rows = runs: row r holds the R samples base + r R .. (element (x, r)); box = 128 bytes x 64 rows.
// Returns false when the view cannot be encoded (alignment); the kernels then take the guarded path everywhere.
bool make_map(CUtensorMap* map, const void* ptr, int elem_bytes, long long base, int R, long long nrows, bool l2_256 = false) {
    memset(map, 0, sizeof(*map));
    EncodeTiledFn fn = encode_fn();
    if (!fn || !ptr || nrows < 1) return false;
    const uintptr_t addr = reinterpret_cast<uintptr_t>(ptr) + (uintptr_t)(base * elem_bytes);   // base <= 0: may lie before the data; never read there
    if (addr & 15) return false;
    if (((long long)R * elem_bytes) & 15) return false;
    if (nrows > 0x7fffffffLL) return false;
    cuuint64_t dims[2] = {(cuuint64_t)R, (cuuint64_t)nrows};
    cuuint64_t strides[1] = {(cuuint64_t)R * (cuuint64_t)elem_bytes};
    cuuint32_t box[2] = {(cuuint32_t)(128 / elem_bytes), (cuuint32_t)kRuns};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const CUresult rc = fn(map, dt, 2, reinterpret_cast<void*>(addr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, l2_256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return rc == CUDA_SUCCESS;
}

long long grid_for(const void* kern, int smem, long long ngroups) {
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kWarps * 32, smem);
    if (occ < 1) occ = 1;
    long long grid = (long long)ct_sm_count() * occ;
    const long long want = (ngroups + kWarps - 1) / kWarps;
    if (grid > want) grid = want;
    if (grid < 1) grid = 1;
    return grid;
}

template <int NSEC, typename InT, int MODE, bool COUNT>
int launch_fwd(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap& im, const CUtensorMap& om, const CtMedianPlan* plan,
               cudaStream_t st) {
    auto kern = ct_filter_fwd_kernel<NSEC, InT, MODE, COUNT>;
    const int smem = kWarps * (2 * kStage + (MODE == 0 ? 2 * kStage : 0)) + kWarps * 16;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const long long grid = grid_for(reinterpret_cast<const void*>(kern), smem, a.ngroups - a.g_first);
    CT_COUNT_LAUNCH();
    kern<<<(unsigned)grid, kWarps * 32, smem, st>>>(im, om, a, k, plan);
    return ct_check_launch("ct_filter_fwd_kernel");
}
template <int NSEC, int D, bool STATS, bool SUMM>
int launch_bwd(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap& om, cudaStream_t st) {
    auto kern = ct_filter_bwd_kernel<NSEC, D, STATS, SUMM>;
    const int smem = kWarps * 2 * kStage;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const long long grid = grid_for(reinterpret_cast<const void*>(kern), smem, a.ngroups - a.g_first);
    CT_COUNT_LAUNCH();
    kern<<<(unsigned)grid, kWarps * 32, smem, st>>>(om, a, k);
    return ct_check_launch("ct_filter_bwd_kernel");
}

#define CT_NSEC_SWITCH(nsec, CALL)                                                              \
    switch (nsec) {                                                                             \
        case 1: { constexpr int NS = 1; return CALL; }                                          \
        case 2: { constexpr int NS = 2; return CALL; }                                          \
        case 3: { constexpr int NS = 3; return CALL; }                                          \
        case 4: { constexpr int NS = 4; return CALL; }                                          \
        case 5: { constexpr int NS = 5; return CALL; }                                          \
    }                                                                                           \
    ct_set_error("filter: nsec must be 1..5, got %d", nsec);                                    \
    return CT_ERR_ARG;

template <typename InT, int MODE>
int dispatch_fwd(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap& im, const CUtensorMap& om, cudaStream_t st,
                 const CtMedianPlan* plan = nullptr) {
    if (sizeof(InT) == 2 && MODE != 0 && a.cw_out) {
        CT_NSEC_SWITCH(k.nsec, (launch_fwd<NS, uint16_t, MODE == 0 ? 1 : MODE, true>(a, k, im, om, plan, st)))
    }
    CT_NSEC_SWITCH(k.nsec, (launch_fwd<NS, InT, MODE, false>(a, k, im, om, plan, st)))
}
template <int D>
int dispatch_bwd(const SeqArgs& a, const CtFilterCoef& k, const CUtensorMap& om, cudaStream_t st) {
    const bool stats = a.st_cnt != nullptr, summ = a.summ != nullptr;
    if (stats && summ) { CT_NSEC_SWITCH(k.nsec, (launch_bwd<NS, D, true, true>(a, k, om, st))) }
    if (stats) { CT_NSEC_SWITCH(k.nsec, (launch_bwd<NS, D, true, false>(a, k, om, st))) }
    if (summ) { CT_NSEC_SWITCH(k.nsec, (launch_bwd<NS, D, false, true>(a, k, om, st))) }
    CT_NSEC_SWITCH(k.nsec, (launch_bwd<NS, D, false, false>(a, k, om, st)))
}

// Decimation factor of the scratch.  Keeping every D-th sample of the forward output and zero-stuffing it in the
// backward pass leaves, at output frequency f, the aliases conj(H(f)) H(f - k fs/D) X(f - k fs/D), k = 1..D-1: the error
// gain is the PRODUCT of the cascade's gains at two frequencies fs/D apart.  D is the largest of 4, 2 for which that
// product stays below eps everywhere (evaluated from the coefficients on the host), else 1.  (8-pole, fs = 4.17 MHz:
// D = 4 up to ~150 kHz, D = 2 up to ~450 kHz, full rate above.)  A pad shorter than the warm-up keeps full rate: the
// held value after the data is then not the settled output.
double cascade_gain(const CtFilterCoef& k, double w) {
    const double cr = cos(w), ci = -sin(w), c2r = cos(2 * w), c2i = -sin(2 * w);   // z^-1, z^-2
    // |1 + z^-1|^order = (2 |cos(w/2)|)^order
    double mag = fabs((double)k.gain) * pow(2.0 * fabs(cos(0.5 * w)), (double)k.order);
    for (int s = 0; s < k.nsec; ++s) {
        const double dr = 1.0 - k.na1[s] * cr - k.na2[s] * c2r, di = -k.na1[s] * ci - k.na2[s] * c2i;
        mag /= sqrt(dr * dr + di * di);
    }
    return mag;
}
int pick_decimation(const CtFilterCoef& k, long long pad, int Hw) {
    if (pad < Hw) return 1;
    static thread_local CtFilterCoef cached_k;
    static thread_local int cached_d = 0;
    if (cached_d && memcmp(&cached_k, &k, sizeof(k)) == 0) return cached_d;
    constexpr int N = 1024;                       // frequencies on [0, 2 pi)
    static thread_local double H[N];
    const double two_pi = 6.283185307179586;
    for (int i = 0; i < N; ++i) H[i] = cascade_gain(k, two_pi * i / N);
    int best = 1;
    for (int D = 4; D >= 2; D >>= 1) {
        double worst = 0.0;
        for (int kk = 1; kk < D; ++kk)
            for (int i = 0; i < N; ++i) { const double v = H[i] * H[(i + kk * (N / D)) % N]; if (v > worst) worst = v; }
        if (worst < 1e-7) { best = D; break; }
    }
    cached_k = k; cached_d = best;
    return best;
}

// Run length for a trace of n samples: long runs amortise the warm-up, but there must be enough
// runs to give every SM a CTA (64 runs per warp, 7 warps per CTA; doubling the warm-up share costs more than a
// half-occupied SM).  Hw <= R always.
int pick_run(long long n, int Hw) {
    const long long target_runs = (long long)ct_sm_count() * kWarps * kRuns;
    static const long long r_max = [] { const char* e = getenv("CT_SEQ_RMAX"); const long long v = e ? atoll(e) : 0; return v >= 256 ? v : 4096; }();
    long long R = r_max;
    while (R > 256 && (n + R - 1) / R < target_runs) R >>= 1;
    while (R < Hw) R <<= 1;
    return (int)R;
}

}  // namespace

extern "C" int64_t ct_filtfilt_workspace_bytes(int64_t n, int64_t pad, int H) {
    const int Hw = (H + kK - 1) / kK * kK;
    const int R = pick_run(n + pad, Hw);
    // one extra group: the run grid may be shifted left by up to a group to align with baseline blocks
    const long long ngroups = (n + pad + (long long)R * kRuns - 1) / ((long long)R * kRuns) + 1;
    return (int64_t)(ngroups * kRuns * (long long)R * 4 + 256);
}

extern "C" int64_t ct_filtfilt_stats_granule(int64_t n, int64_t pad, int H) {
    const int Hw = (H + kK - 1) / kK * kK;
    return (int64_t)pick_run(n + pad, Hw) * kRuns;
}

extern "C" int ct_filter_decimation(const CtFilterCoef* coef, int64_t pad, int H) {
    if (!coef) { ct_set_error("filter_decimation: null coefficients"); return CT_ERR_ARG; }
    return pick_decimation(*coef, pad, (H + kK - 1) / kK * kK);
}

/* float2 entries the chunk-extrema array of ct_filter_backward needs (one per 64 output samples of the run grid) */
extern "C" int64_t ct_filter_summary_count(int64_t n, int64_t pad, int H) {
    return ct_filtfilt_workspace_bytes(n, pad, H) / 4 / kK;
}

namespace {

struct Plan { int Hw, R; long long G, base, n1, ng_fwd, ng_bwd, g_right; };
// Run grid of a trace of n samples (+ pad): groups of G = 64 R samples starting at `base` <= 0 with
// base = origin (mod G), so that groups never straddle a baseline block counted from `origin`.
Plan make_plan(long long n, long long pad, int H, long long origin) {
    Plan p;
    p.Hw = (H + kK - 1) / kK * kK;
    p.n1 = n + pad;
    p.R = pick_run(p.n1, p.Hw);
    p.G = (long long)p.R * kRuns;
    p.base = -((p.G - origin % p.G) % p.G);
    p.ng_fwd = (p.n1 - p.base + p.G - 1) / p.G;
    p.ng_bwd = (n - p.base + p.G - 1) / p.G;
    p.g_right = (n - p.base) / p.G;                       // first group that sees positions >= n (the right pad)
    return p;
}
void init_args(SeqArgs& a) {
    memset(&a, 0, sizeof(a));
    a.st_block = 1; a.mask = 0xffffu; a.scale = 1.f;
}
int check_ws(const void* workspace, int64_t workspace_bytes, int64_t n, int64_t pad, int H) {
    if (!workspace || workspace_bytes < ct_filtfilt_workspace_bytes(n, pad, H) || (reinterpret_cast<uintptr_t>(workspace) & 63)) {
        ct_set_error("filter: workspace missing, too small or not 64-byte aligned"); return CT_ERR_ARG;
    }
    return CT_OK;
}
// x' = value - sub with an INTEGER constant inside the kernel (exact in the byte-permute conversion): the fractional
// part of `sub` (0 or 0.5 for a median of codes) moves into the pad value and the output offset (the cascade's DC
// gain is 1: filtfilt(x + f) = filtfilt(x) + f).
void split_sub(SeqArgs& a, float sub, float pad_x) {
    const float fl = floorf(sub);
    a.isub = (int)fl;
    a.fsub = sub;
    a.pad_x = pad_x + (sub - fl);
}

}  // namespace

// Forward pass into the scratch.  in_kind: 0 = uint16 codes, 1 = float32 samples.  part: 0 = whole
// trace, 1 = only the groups whose result depends on pad_x (the two ends of the trace), 2 = streaming.
// counts9 != NULL (uint16 only, part 0/2): also tally the window count for the exact median.
// plan_dev != NULL (uint16 only): sub and cw_lo are read from it on the device, the values passed here are ignored.
int ct_filter_forward_seq(const void* in, int in_kind, int64_t n, int64_t pad, float sub, uint16_t mask, float pad_x,
                          const CtFilterCoef* coef, int H, int64_t origin, int part, uint32_t cw_lo, uint32_t cw_step,
                          int64_t cw_begin, int64_t cw_end, uint64_t* counts9, int64_t from_pos, int64_t to_pos,
                          void* workspace, int64_t workspace_bytes, const float* pad_x_dev, const CtMedianPlan* plan_dev,
                          cudaStream_t st) {
    int rc = check_ws(workspace, workspace_bytes, n, pad, H); if (rc) return rc;
    const Plan p = make_plan(n, pad, H, origin);
    SeqArgs a; init_args(a);
    a.in = in; a.n_in = n; a.mask = mask; a.Hw = p.Hw; a.R = p.R; a.base = p.base;
    if (plan_dev) { a.pad_x = pad_x; cw_lo = 0; }        // the kernel does the rest of split_sub and of cw_c
    else if (in_kind == 0) split_sub(a, sub, pad_x);
    else { a.fsub = sub; a.pad_x = pad_x; }
    a.out = reinterpret_cast<float*>(workspace);
    a.pad_x_dev = part == 1 ? pad_x_dev : nullptr;
    a.scratch_floats = (ct_filtfilt_workspace_bytes(n, pad, H) - 256) / 4;
    if (counts9 && part != 1 && in_kind == 0) {
        if (!cw_step || (cw_step & (cw_step - 1))) { ct_set_error("filter: window step must be a power of two"); return CT_ERR_ARG; }
        if ((cw_lo & (cw_step - 1)) || (mask & (cw_step - 1))) {     // the tally's nibble index 4 (code - lo) / step
            ct_set_error("filter: the window's first code and every masked code must be multiples of the window step");
            return CT_ERR_ARG;
        }
        if (cw_step > 4) { ct_set_error("filter: the fused window count needs a window step <= 4 (ADC of 14 bits or more)"); return CT_ERR_UNSUPPORTED; }
        a.cw_k = 4u / cw_step; a.cw_c = 0u - (0x4B000000u + cw_lo) * a.cw_k; a.cw_out = (unsigned long long*)counts9;
        a.cw_p0 = cw_begin < 0 ? 0 : cw_begin; a.cw_p1 = cw_end > n ? n : cw_end;
    }
    const int D = pick_decimation(*coef, pad, p.Hw);
    a.scale = (float)D; a.offset = 0.f;
    CUtensorMap im, om;
    memset(&om, 0, sizeof(om));
    a.tma_in = make_map(&im, in, in_kind ? 4 : 2, p.base, p.R, p.ng_fwd * kRuns, true) ? 1 : 0;
    // the work counter lives in the last 256 bytes of the workspace (never part of the scratch)
    a.next_group = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(workspace) + ct_filtfilt_workspace_bytes(n, pad, H) - 256);
    auto go = [&](const SeqArgs& x) {
        cudaMemsetAsync(x.next_group, 0, 8, st);
        if (in_kind) {
            if (D == 4) return dispatch_fwd<float, 4>(x, *coef, im, om, st);
            if (D == 2) return dispatch_fwd<float, 2>(x, *coef, im, om, st);
            return dispatch_fwd<float, 1>(x, *coef, im, om, st);
        }
        if (D == 4) return dispatch_fwd<uint16_t, 4>(x, *coef, im, om, st, plan_dev);
        if (D == 2) return dispatch_fwd<uint16_t, 2>(x, *coef, im, om, st, plan_dev);
        return dispatch_fwd<uint16_t, 1>(x, *coef, im, om, st, plan_dev);
    };
    if (part == 0) { a.g_first = 0; a.ngroups = p.ng_fwd; return go(a); }
    if (part == 2) {
        // streaming: the groups whose input [.., group end) lies below to_pos (all remaining ones once to_pos >= n)
        // and that were not covered by the previous call (which ended at from_pos)
        auto done = [&](long long pos) { return pos >= n ? p.ng_fwd : (pos <= p.base ? 0 : (pos - p.base) / p.G); };
        a.g_first = done(from_pos); a.ngroups = done(to_pos);
        return a.g_first < a.ngroups ? go(a) : CT_OK;
    }
    a.g_first = 0; a.ngroups = p.ng_fwd < 1 ? p.ng_fwd : 1;            // left end: group 0
    rc = go(a); if (rc) return rc;
    if (p.g_right >= 1 || p.ng_fwd > 1) {                                 // right end: groups that reach the right pad
        a.g_first = p.g_right > 1 ? p.g_right : 1; a.ngroups = p.ng_fwd;
        if (a.g_first < a.ngroups) rc = go(a);
    }
    return rc;
}

// Backward pass scratch -> out = offset + scale * y (+ optional fused baseline block sums and chunk extrema).
int ct_filter_backward_seq(int64_t n, int64_t pad, float sub, float scale, float offset, const CtFilterCoef* coef, int H,
                           int64_t origin, float* out, const void* workspace, int64_t workspace_bytes,
                           const CtFilterStats* stats, float* summaries, cudaStream_t st) {
    int rc = check_ws(workspace, workspace_bytes, n, pad, H); if (rc) return rc;
    const Plan p = make_plan(n, pad, H, origin);
    SeqArgs b; init_args(b);
    b.in = workspace; b.n_in = p.n1; b.out = out; b.n_out = n; b.scale = scale;
    b.offset = offset - scale * (sub - floorf(sub));      // see split_sub: the kernel subtracted floor(sub)
    b.Hw = p.Hw; b.R = p.R; b.base = p.base; b.scratch_runs = p.ng_fwd * kRuns; b.ngroups = p.ng_bwd;
    b.summ = reinterpret_cast<float2*>(summaries);
    b.scratch_floats = (ct_filtfilt_workspace_bytes(n, pad, H) - 256) / 4;
    b.summ_count = ct_filter_summary_count(n, pad, H);
    if (summaries && (reinterpret_cast<uintptr_t>(summaries) & 31)) { ct_set_error("filter: chunk extrema must be 32-byte aligned"); return CT_ERR_ARG; }
    if (stats) {
        if (stats->block <= 0 || stats->block % p.G || stats->origin != origin || !stats->cnt || !stats->s1 || !stats->s2) {
            ct_set_error("filter: fused block statistics need block %% %lld == 0 and the grid origin (block = %lld)", p.G,
                         (long long)stats->block);
            return CT_ERR_ARG;
        }
        if (stats->block < 65536) {       // the epilogue's 32-bit partial sums: |q| < 2^31 / sqrt(block) must stay below 2^23
            ct_set_error("filter: fused block statistics need blocks of at least 65536 samples (got %lld)", (long long)stats->block);
            return CT_ERR_UNSUPPORTED;
        }
        const long long nb = (n - stats->origin + stats->block - 1) / stats->block;
        if (nb > 0) {
            cudaMemsetAsync(stats->cnt, 0, nb * 8, st); cudaMemsetAsync(stats->s1, 0, nb * 8, st); cudaMemsetAsync(stats->s2, 0, nb * 8, st);
        }
        b.st_origin = stats->origin; b.st_block = stats->block; b.st_min = stats->bmin; b.st_max = stats->bmax;
        b.st_scale = ldexpf(1.f, stats->shift); b.st_nc0s = -ldexpf(stats->c0, stats->shift);
        b.st_cnt = (long long*)stats->cnt; b.st_s1 = (long long*)stats->s1; b.st_s2 = (long long*)stats->s2;
    }
    CUtensorMap om;
    b.tma_out = make_map(&om, out, 4, p.base, p.R, p.ng_bwd * kRuns) ? 1 : 0;
    b.next_group = reinterpret_cast<unsigned long long*>(const_cast<char*>(reinterpret_cast<const char*>(workspace)) +
                                                        ct_filtfilt_workspace_bytes(n, pad, H) - 256) + 1;
    cudaMemsetAsync(b.next_group, 0, 8, st);
    const int D = pick_decimation(*coef, pad, p.Hw);
    if (D == 4) return dispatch_bwd<4>(b, *coef, om, st);
    if (D == 2) return dispatch_bwd<2>(b, *coef, om, st);
    return dispatch_bwd<1>(b, *coef, om, st);
}

// One call: forward (+ backward).  stats (may be NULL): fused baseline block sums of the output.
int ct_filtfilt_seq(const void* in, int in_kind, int64_t n, int64_t pad, float sub, uint16_t mask, float scale,
                    float offset, const CtFilterCoef* coef, int H, int forward_only, float* out, void* workspace,
                    int64_t workspace_bytes, const CtFilterStats* stats, cudaStream_t st) {
    if (forward_only) {
        if (stats) { ct_set_error("filter: block statistics are fused into the zero-phase path only"); return CT_ERR_UNSUPPORTED; }
        SeqArgs a; init_args(a);
        a.in = in; a.n_in = n; a.mask = mask;
        if (in_kind == 0) split_sub(a, sub, 0.f); else { a.fsub = sub; a.pad_x = 0.f; }
        a.scale = scale; a.offset = in_kind == 0 ? offset - scale * (sub - floorf(sub)) : offset;
        a.Hw = (H + kK - 1) / kK * kK; a.R = pick_run(n, a.Hw);
        a.ngroups = (n + (long long)a.R * kRuns - 1) / ((long long)a.R * kRuns);
        a.out = out; a.n_out = n;
        CUtensorMap im, om;
        a.tma_in = make_map(&im, in, in_kind ? 4 : 2, 0, a.R, a.ngroups * kRuns) ? 1 : 0;
        a.tma_out = make_map(&om, out, 4, 0, a.R, a.ngroups * kRuns) ? 1 : 0;
        return in_kind ? dispatch_fwd<float, 0>(a, *coef, im, om, st) : dispatch_fwd<uint16_t, 0>(a, *coef, im, om, st);
    }
    const int64_t origin = stats ? stats->origin : 0;
    int rc = ct_filter_forward_seq(in, in_kind, n, pad, sub, mask, 0.f, coef, H, origin, 0, 0, 1, 0, 0, nullptr, 0, 0, workspace,
                                   workspace_bytes, nullptr, nullptr, st);
    if (rc) return rc;
    return ct_filter_backward_seq(n, pad, in_kind == 0 ? sub : 0.f, scale, offset, coef, H, origin, out, workspace, workspace_bytes,
                                  stats, nullptr, st);
}
