/* cusumtools_b200 — C ABI of the B200-native raw-trace hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference
 * (shadowk29/cusumtools) is pure Python with no FFI of its own; its de-facto operator
 * boundary for this path is four library calls plus file formats (SURVEY.md section 8b).
 * Each entry point below names the reference call site it replaces.  A maintainer binds
 * these with ctypes (see INTEGRATION.md; cusumtools_b200/_lib.py is that binding).
 *
 * Conventions
 *   - every pointer except `coef`, `sign`-less scalars and `ct_last_error` results is a
 *     DEVICE pointer owned by the caller; the library never frees or retains it;
 *   - `stream` is a cudaStream_t (0 = default stream); all work is enqueued on it and no
 *     entry point synchronises the device;
 *   - return value 0 = ok, negative = error (CT_ERR_*), message via ct_last_error();
 *   - 64-bit sample counts everywhere (a 1-hour trace has 1.5e10 samples).
 */
#ifndef CUSUMTOOLS_B200_H
#define CUSUMTOOLS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CT_ABI_VERSION 2
#define CT_MAX_SECTIONS 5

/* Filter coefficients as the kernel consumes them (built on the host in float64 by
 * cusumtools_b200/design.py from the same Bessel design the reference requests with
 * scipy.signal.bessel(order, Wn, 'low') at plot-trace.py:317):
 *   H(z) = gain (1 + z^-1)^order / prod_s (1 - na1[s] z^-1 - na2[s] z^-2)
 *   fir[k] = gain * C(order, k), k = 0..order (zero beyond): the numerator as one binomial FIR
 *   ss[s]  = steady-state output of all-pole section s for a unit constant at the cascade input
 *   gain   = prod_s (1 - na1[s] - na2[s]) / 2^order, evaluated from the float32-rounded na1/na2: DC gain exactly 1 */
typedef struct CtFilterCoef {
    int32_t nsec;
    int32_t order;
    float na1[CT_MAX_SECTIONS], na2[CT_MAX_SECTIONS];
    float ss[CT_MAX_SECTIONS];
    float fir[2 * CT_MAX_SECTIONS + 1];
    float gain;
} CtFilterCoef;

int ct_version(void);
const char* ct_last_error(void);                  /* thread-local, never NULL */
uint64_t ct_launch_count(void);                   /* kernels launched by this library so far */
void ct_launch_count_reset(void);
int ct_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* smem_optin);

/* ---- stage 1: dequantise + median pad + zero-phase Bessel -------------------------
 * Replaces App.scale_raw_data + App.filter_data (plot-trace.py:272-287, 313-320):
 *   out[i] = pad_value + alpha * filtfilt(code - median_code)[i],  i in [0, n)
 * with the reference's boundary semantics (constant pad of `pad` samples each side,
 * steady-state initial conditions).  raw codes are masked with `mask` first
 * (plot-trace.py:281-282).  forward_only != 0 gives the causal pass only (scipy.signal.lfilter
 * with zi = lfilter_zi*pad_value), the primitive filtfilt is built from.
 *   Two lane-sequential passes staged with TMA; H = IIR warm-up per run (any value, rounded up to
 *   ct_filter_seq_tile()); workspace = ct_filtfilt_workspace_bytes(n, pad, H) bytes of device scratch
 *   (64-byte aligned) for the forward output, unused if forward_only.  The scratch keeps every D-th
 *   forward sample, D = ct_filter_decimation(coef, pad, H) in {1, 2, 4}, chosen from the cascade's
 *   own stop band so that the aliasing error stays below 1e-7 of the signal.                    */
/* Optional fusion of ct_block_stats_f32 into the zero-phase filter: the final
 * samples are tallied on their way out, which saves the separate 4 B/sample pass.  The block
 * grid starts at output sample `origin` (samples before it are not tallied; time shards put
 * their left halo there); `block` must be a multiple of ct_filtfilt_stats_granule(n, pad, H).
 * cnt/s1/s2: int64[ceil((n - origin)/block)] device arrays, zeroed by the call.          */
typedef struct CtFilterStats {
    int64_t origin, block;
    float bmin, bmax, c0;
    int32_t shift;
    int64_t* cnt; int64_t* s1; int64_t* s2;
} CtFilterStats;

int ct_filter_seq_tile(void);
int ct_filter_decimation(const CtFilterCoef* coef, int64_t pad, int H);
int64_t ct_filtfilt_stats_granule(int64_t n, int64_t pad, int H);
int64_t ct_filtfilt_workspace_bytes(int64_t n, int64_t pad, int H);
int ct_filtfilt_u16(const uint16_t* raw, int64_t n, int64_t pad, float median_code, uint16_t mask,
                    float alpha, float pad_value, const CtFilterCoef* coef, int H,
                    int forward_only, float* out, void* workspace, int64_t workspace_bytes,
                    const CtFilterStats* stats, void* stream);
/* Same for already-dequantised float32 input (.bin traces, print_trace.py:33,
 * noise-fit.py:90; multi-gain file series, plot-trace.py:252-269):
 *   out = pad_value + filtfilt(x - pad_value).                                         */
int ct_filtfilt_f32(const float* x, int64_t n, int64_t pad, float pad_value, const CtFilterCoef* coef,
                    int H, int forward_only, float* out, void* workspace, int64_t workspace_bytes,
                    const CtFilterStats* stats, void* stream);

/* The two passes as separate calls, for callers that know the median only
 * approximately when the forward pass starts (streaming loads; fusing the exact count into the
 * pass that reads every code anyway).  With DC gain exactly 1,
 *     filtfilt(code - m) + m == filtfilt(code - c) + c      for ANY constant c,
 * provided the pad holds m - c instead of 0.  So the forward pass may subtract an estimate c
 * (`sub_code`) with pad_x = 0; it can tally, on the side, the window counts that pin the exact
 * median m (counts9: as ct_count_window_u16, window_step <= 4, window_lo and every masked code multiples of window_step,
 * else CT_ERR_ARG and counts9 untouched; zeroed by the caller); if m != c the caller re-runs
 * only the groups the pad influences (`part` = 1, pad_x = m - c) and then runs the backward
 * pass with the same sub_code and offset = value(sub_code).  `origin` (>= 0) aligns the run grid with
 * baseline blocks counted from that output sample; both passes must get the same value.  Only codes at
 * positions [count_begin, count_end) are tallied (a time shard counts its owned samples, not its halos).
 * part = 2 streams the pass while the codes are still arriving: each call processes the groups
 * whose input lies below to_pos and that the previous call (which ended at from_pos) did not.
 * chunk_minmax (may be NULL): float[2 * ct_filter_summary_count(n, pad, H)], 32-byte aligned; entry c
 * receives (min, max) of the output samples [64 c - shift, 64 c - shift + 64), shift = (G - origin % G) % G with
 * G = ct_filtfilt_stats_granule (0 when origin is 0): what ct_detect_f32 needs to classify whole chunks
 * without re-reading the trace.  Entries of chunks that are not entirely inside [0, n) are unspecified. */
int64_t ct_filter_summary_count(int64_t n, int64_t pad, int H);
int ct_filter_forward_u16(const uint16_t* raw, int64_t n, int64_t pad, float sub_code, uint16_t mask, float pad_x,
                          const CtFilterCoef* coef, int H, int64_t origin, int part, uint32_t window_lo,
                          uint32_t window_step, int64_t count_begin, int64_t count_end, uint64_t* counts9, int64_t from_pos,
                          int64_t to_pos, void* workspace, int64_t workspace_bytes, void* stream);
/* The same step without a host round trip between the passes (the GPU would idle from the end of the forward pass until
 * the host has turned the counts into the median and launched the rest):
 *   ct_median_verify: ONE thread evaluates the counts (uint64[1 + nbins]: #codes < lo, #codes == lo + i*step; summed over
 *     the ranks by the caller if there are several) for the order statistics k1 <= k2 (0-based ranks of the two middle
 *     codes) and leaves them in `result` (device memory) with pad_x = (code1 + code2) / 2 - sub_code;
 *     status 0 = found, 1 = the window lies above the median, 2 = below (code / pad fields 0: the caller re-counts);
 *   ct_filter_forward_ends_u16: `part` = 1 of ct_filter_forward_u16 with the pad read from `result->pad_x` on the device;
 *     its CTAs return at once when it is 0 (the estimate was the median). */
typedef struct CtMedianResult {
    uint32_t code1, code2;   /* the two middle order statistics of the masked codes */
    float pad_x;             /* median - sub_code */
    uint32_t status;
} CtMedianResult;
int ct_median_verify(const uint64_t* counts9, int nbins, int64_t k1, int64_t k2, uint32_t lo, uint32_t step, float sub_code,
                     CtMedianResult* result, void* stream);
int ct_filter_forward_ends_u16(const uint16_t* raw, int64_t n, int64_t pad, float sub_code, uint16_t mask,
                               const float* pad_x_dev, const CtFilterCoef* coef, int H, int64_t origin, void* workspace,
                               int64_t workspace_bytes, void* stream);
int ct_filter_backward(int64_t n, int64_t pad, float sub_code, float scale, float offset, const CtFilterCoef* coef, int H,
                       int64_t origin, float* out, const void* workspace, int64_t workspace_bytes, const CtFilterStats* stats,
                       float* chunk_minmax, void* stream);

/* Exact global median of the masked codes, the value np.pad(mode='median') needs
 * (plot-trace.py:319): a strided-sample histogram to locate it and an exact count of
 * the codes below / inside a window of 8 codes {lo + i*step} to verify it.
 *   hist65536: uint32[65536], caller-zeroed; counts9: uint64[9], caller-zeroed.
 * The window counts need step a power of two and lo and mask multiples of it (mask & (step - 1) == 0: every masked
 * code is some lo + i*step or outside the window); any other step, lo or mask returns CT_ERR_ARG with counts9 untouched.
 * ct_count_window4_u16 counts only the first four window codes (counts9[5..8] untouched): the
 * cheaper first attempt when the estimate comes from a sample of the whole trace.         */
int ct_hist_sampled_u16(const uint16_t* raw, int64_t n, int64_t stride, uint16_t mask,
                        uint32_t* hist65536, void* stream);

/* Rank search in the (summed) histogram on the device: out3[0] = first bin whose cumulative count reaches half the total
 * (the sampled median), out3[1] = its count, out3[2] = the total.  hist65536: uint32[65536], or int64[65536] (is_int64)
 * after an all_reduce over ranks. */
int ct_hist_rank(const void* hist65536, int is_int64, int64_t* out3, void* stream);
int ct_count_window_u16(const uint16_t* raw, int64_t n, uint16_t mask, uint32_t lo, uint32_t step,
                        uint64_t* counts9, void* stream);
int ct_count_window4_u16(const uint16_t* raw, int64_t n, uint16_t mask, uint32_t lo, uint32_t step,
                         uint64_t* counts9, void* stream);

/* ---- stage 2: baseline statistics + threshold/hysteresis detection ---------------
 * No reference implementation exists; semantics per plot-trace.py:379-414, definition in
 * oracle/events_oracle.py.  Block sums are exact int64 sums of
 * q = rint((y - c0) * 2^shift) over samples with bmin <= y <= bmax.                   */
int ct_block_stats_f32(const float* y, int64_t n, int64_t block, float bmin, float bmax, float c0,
                       int shift, int64_t* cnt, int64_t* s1, int64_t* s2, void* stream);
/* Baseline table + detector thresholds from the block sums, entirely on the device (the
 * rows of baseline.csv and the two dashed lines of plot-trace.py:408-411):
 *   mean = c0 + (s1/cnt) 2^-shift, std = sqrt(max(s2/cnt - (s1/cnt)^2, 0)) 2^-shift in
 *   individually rounded float64 operations; blocks with cnt < min_count inherit the nearest
 *   earlier valid block; sign = sign(mean); t_start = (float)(mean - sign*threshold*std);
 *   t_end = (float)(mean - sign*(threshold - hysteresis)*std).  status[0] = 1 if no block
 *   is valid (nothing else is written then).  All arrays have nb entries.                */
int ct_baseline_finalize(const int64_t* cnt, const int64_t* s1, const int64_t* s2, int64_t nb, float c0, int shift,
                         int64_t min_count, double threshold, double hysteresis, double* mean, double* stdev,
                         int32_t* sign, float* t_start, float* t_end, int32_t* status, void* stream);
int ct_detect_run(void);                          /* `block` must be a multiple of this */
int64_t ct_detect_workspace_bytes(int64_t n);
/* starts/ends: int64[capacity] in time order; counts2 = {n_starts, n_ends} (may exceed
 * capacity: nothing is written past it).  With state_in == 0 event i is
 * [starts[i], ends[i]) for i < n_ends and starts[n_ends] (if any) is still open.
 * chunk_minmax (may be NULL): the (min, max) pairs ct_filter_backward left for the 64-sample chunks of y,
 * entry c covering samples [64 c - minmax_shift, 64 c - minmax_shift + 64); whole chunks are then classified
 * against the block's lines and only chunks that hold a crossing are read from y (same result).   */
int ct_detect_f32(const float* y, int64_t n, int64_t block, const int32_t* sign, const float* t_start,
                  const float* t_end, int state_in, const float* chunk_minmax, int64_t minmax_shift, void* workspace,
                  int64_t workspace_bytes, int64_t* starts, int64_t* ends, int64_t capacity, uint64_t* counts2, void* stream);

/* Event windows handed to CUSUM+ and the rate.csv `type` code (0 accepted, 2 shorter than
 * minpoints, 3 longer than maxpoints, 4 padding leaves the trace or overlaps a neighbour;
 * plot-trace.py:354-357 treats type > 1 as rejected), computed on the device from the
 * detector's own counters so no host round trip separates detection from CUSUM+.
 * Event i is [starts[i], ends[i]) for i < min(counts2[0], counts2[1], capacity); the events
 * with pos_lo <= start < pos_hi are kept (time shards: the rank whose owned range holds the
 * start owns the event; detection itself starts in the left halo so that the state at the
 * first owned sample is right).  They are the index range [i0, i0 + count) of starts/ends;
 * win = [start - padding, end + padding) and type are written compacted (index i - i0);
 * out2 = {count, i0}.                                                                    */
int ct_event_windows(const int64_t* starts, const int64_t* ends, const uint64_t* counts2, int64_t capacity,
                     int64_t n_total, int64_t pos_lo, int64_t pos_hi, int64_t padding, int64_t minpoints, int64_t maxpoints,
                     int64_t* win_start, int64_t* win_end, int32_t* type, int64_t* out2, void* stream);

/* ---- stage 3: batched per-event CUSUM+ level segmentation -----------------------
 * No reference implementation exists (readevents.py:843-846,1297-1306 only consumes the
 * level lists); definition in oracle/events_oracle.py::cusum_event (two-sided CUSUM,
 * SURVEY.md Appendix C, all reductions in exact integers).  Event e is the window
 * y[win_start[e] : win_end[e]) of the filtered trace; events with type[e] != 0 are
 * skipped (type may be NULL).  Outputs per event: n_levels, edges[max_levels+1] (sample
 * offsets inside the window, edges[0] = 0, edges[n_levels] = length, unused = -1),
 * level mean / population std in pA (float64), overflow flag (more jumps than
 * max_levels-1).  workspace: ct_cusum_workspace_bytes(n_events) bytes of device scratch
 * (16-byte aligned; the library keeps no device state of its own).  Windows of up to 16384
 * samples are segmented one event per lane (y 16-byte aligned, batches of >= 16384 events),
 * everything else one event per warp.  Domain of the definition: |y - y[win_start[e]]| < 65536 pA
 * inside a window (samples are quantised to 1/64 pA relative to the window's first sample).   */
int64_t ct_cusum_workspace_bytes(int64_t n_events);
int ct_cusum_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                   const int32_t* type, int64_t n_events, float delta, float h, int max_levels,
                   int32_t* n_levels, int32_t* edges, double* level_mean, double* level_std,
                   uint8_t* overflow, void* workspace, int64_t workspace_bytes, void* stream);
/* Same with the event count read from device memory (n_events_dev[0], clamped to capacity):
 * the output arrays must hold `capacity` rows; rows at or beyond the count are not written. */
int ct_cusum_batch_dev(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                       const int32_t* type, const int64_t* n_events_dev, int64_t capacity, float delta, float h,
                       int max_levels, int32_t* n_levels, int32_t* edges, double* level_mean, double* level_std,
                       uint8_t* overflow, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- stage 3b: step-response fit of short events (type 1) ---------------------------
 * No reference implementation exists: readevents.py:1334-1337 reads a type-1 event file with the four columns
 * time, current, cusum, stepfit, and events.csv carries rc_const1_us / rc_const2_us (writer convention:
 * cusumtools_b200/writer.py, type 1 = step-response fit, 7 = step fit failed, rate.csv only).  Definition of record:
 * oracle/stepfit_oracle.py.  For window sample t (window = [win_start, win_end)) and p = (i0, a, u1, u2, tau1, tau2):
 *   f(t) = i0 - a (1 - exp(-(t-u1)/tau1)) H(t-u1) + a (1 - exp(-(t-u2)/tau2)) H(t-u2),   H(s) = [s >= 0].
 * ct_stepfit_select turns the accepted events (type 0) shorter than `stepfit_samples` (event length =
 * win_end - win_start - 2 padding) into type 1; it must run BEFORE ct_cusum_batch_dev, so that CUSUM+ skips them.
 * n_events_dev may be NULL (all `capacity` rows).                                                                 */
#define CT_STEPFIT_MAX_WINDOW 8192                /* longest window ct_stepfit_batch fits (longer: type 7) */
int ct_stepfit_select(const int64_t* win_start, const int64_t* win_end, int32_t* type, const int64_t* n_events_dev,
                      int64_t capacity, int64_t padding, int64_t stepfit_samples, void* stream);
/* Levenberg-Marquardt fit of every type-1 event from the initial guess i0 = mean of the first and last `padding`
 * samples, a = i0 - mean of the rest, u1 = padding, u2 = n - padding, tau1 = tau2 = tau0 (samples), at most
 * `max_iters` LM trials.  A valid fit writes its level rows (n_levels = 3, edges = {0, ceil u1, ceil u2, n},
 * mean = {i0, i0 - a, i0}, std = rms of the residual over each level); an invalid fit or a window it rejects (outside
 * [0, n_total), not longer than 2 padding, longer than CT_STEPFIT_MAX_WINDOW) sets type 7, n_levels = 0 and the edge
 * row to -1.  params6 [capacity][6] (i0 and a in pA, the rest in samples), cost (sum of squared residuals, pA^2) and
 * iters (LM trials: the initial evaluation and every trial after it, including those never evaluated because the
 * matrix was not positive definite or the trial point left the domain tau > 0, u1 < u2) are written for every row
 * below the count, zero for events that are not type 1 and for rejected windows.  It must run AFTER
 * ct_cusum_batch_dev, which writes n_levels = 0 for every event whose type is not 0.                               */
int ct_stepfit_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end, int32_t* type,
                     const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0, int max_iters, int max_levels,
                     double* params6, double* cost, int32_t* iters, int32_t* n_levels, int32_t* edges, double* level_mean,
                     double* level_std, void* stream);

/* Fallback of the events CUSUM+ leaves without a sub-level (the events ct_event_columns would report as type 5):
 * ct_stepfit_fallback_select runs AFTER ct_cusum_batch_dev (or after the level rows were zeroed when CUSUM+ is off) and
 * marks every row below the count with type 0, overflow 0 and n_levels < 3: type 1 if its window is at most
 * CT_STEPFIT_MAX_WINDOW samples, else CT_TYPE_STEPFIT_LONG.  No other row changes.  n_events_dev may be NULL.
 * ct_stepfit_long_batch takes the arguments of ct_stepfit_batch and fits the rows of type CT_TYPE_STEPFIT_LONG with one
 * CTA per event, with the same initial guess, LM loop, stop tests, validity rule and level rows; each such row becomes
 * type 1 or 7 (a window outside [0, n_total), not longer than 2 padding or longer than CT_STEPFIT_LONG_MAX_WINDOW: type 7,
 * n_levels = 0, edge row -1, zero params / cost / iters).  It does not touch any row of another type.
 * row_counter: one int64 of device scratch (the CTAs claim rows from it; reset by the call), not shared with a call that
 * may run at the same time.
 * Launch order: ct_stepfit_batch, then ct_stepfit_long_batch.  ct_stepfit_batch zeroes the params row of every row
 * that is not type 1, which the long fit then overwrites; the other way round, ct_stepfit_batch would take the long
 * rows that had just become type 1 and reject their windows as too long.
 * Type codes of the step: 1 step-response fit (short events, or fallback), 5 (ct_event_columns) accepted but no
 * sub-level, 7 step fit failed (an event of any length), 8 = CT_TYPE_STEPFIT_LONG: long fit pending, internal to the
 * step (never left in a result).                                                                                    */
#define CT_TYPE_STEPFIT_LONG 8
#define CT_STEPFIT_LONG_MAX_WINDOW 131072         /* longest window ct_stepfit_long_batch fits; t - k exact in float32 */
int ct_stepfit_fallback_select(const int32_t* n_levels, const uint8_t* overflow, const int64_t* win_start,
                               const int64_t* win_end, int32_t* type, const int64_t* n_events_dev, int64_t capacity,
                               void* stream);
int ct_stepfit_long_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end, int32_t* type,
                          const int64_t* n_events_dev, int64_t capacity, int64_t padding, float tau0, int max_iters,
                          int max_levels, double* params6, double* cost, int32_t* iters, int32_t* n_levels, int32_t* edges,
                          double* level_mean, double* level_std, int64_t* row_counter, void* stream);

/* Intra-event threshold crossings (rate.csv intra_crossing_times_us / events.csv intra_crossings;
 * consumer: readevents.py:1340-1343,1363-1367, summary.txt keys intra_threshold / intra_hysteresis
 * readevents.py:73-79).  The detector's automaton over each event window with the lines
 * t_start / t_end (per baseline block, built from intra_threshold / intra_hysteresis by
 * ct_baseline_finalize) of the block holding ev_start; starts outside, an open crossing ends at
 * the window end.  count[i] = crossings of event i; pairs[i][2k], pairs[i][2k+1] = start / end
 * sample relative to win_start[i] for k < min(count[i], max_pairs).  n_events_dev may be NULL. */
int ct_intra_crossings_f32(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                           const int64_t* ev_start, int64_t n_events, const int64_t* n_events_dev, int64_t block,
                           int64_t n_blocks, const int32_t* sign, const float* t_start, const float* t_end,
                           int32_t max_pairs, int32_t* count, int32_t* pairs, void* stream);

/* Minimum and maximum sample of every event window (max_deviation_pA of events.csv,
 * mosaicConverter.py:105 / readevents.py:1499); n_events_dev may be NULL.                  */
int ct_event_extrema_f32(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                         int64_t n_events, const int64_t* n_events_dev, float* xmin, float* xmax, void* stream);

/* Derived per-event statistics: the non-level columns of events.csv that mosaicConverter.py:72-154 computes from an
 * event's level list (readevents.py:1470-1508 names them), one thread per event from the level table of ct_cusum_batch:
 *   cols12[e] = { baseline_before, baseline_after, effective_baseline, sub-level duration (samples), average_blockage,
 *                 max_blockage, length of its level (samples), min_blockage, length of its level, residual,
 *                 max_deviation, 0 }                                (pA; conventions: cusumtools_b200/writer.py)
 *   type_out[e] = type[e], or 5 (accepted but CUSUM+ found no sub-level) / 6 (level overflow); type 1 (step-response
 *   fit, level rows from ct_stepfit_batch) is treated as type 0; rows of events with type_out > 1 are zero.  xmin / xmax: ct_event_extrema_f32.  type and n_events_dev may be NULL.                */
int ct_event_columns(const int32_t* n_levels, const int32_t* edges, const double* level_mean, const double* level_std,
                     const int32_t* type, const uint8_t* overflow, const float* xmin, const float* xmax, int64_t n_events,
                     const int64_t* n_events_dev, int max_levels, double* cols12, int32_t* type_out, void* stream);

/* ---- stage 4: Welch PSD ------------------------------------------------------------
 * Replaces scipy.signal.welch(x, fs, nperseg=L) as called at plot-trace.py:442,
 * noise-fit.py:92 (use_abs != 0: welch(|x|)), legacy/minimal_psd.py:255: periodic Hann,
 * hop L/2, tail dropped, per-segment mean removal.  L = nperseg must be a power of two.
 * acc[k] (float64, k = 0..L/2) receives sum over segments of |rfft(w (x_s - mean x_s))[k]|^2;
 * the caller divides by nseg * fs * sum(w^2) = nseg * fs * 3L/8 and doubles bins 1..L/2-1.
 * `shift` is any constant near the signal mean (subtracted before the float32 FFT, exactly
 * compensated); `batch` segments are transformed per launch pair (intermediate
 * batch * L/2 * 8 bytes in the workspace for L > 2^14; larger batches amortise the per-CTA set-up;
 * shorter segments need no intermediate).  256 <= L <= 2^23.                            */
int64_t ct_welch_workspace_bytes(int32_t nperseg, int32_t batch);
int ct_welch_f32(const float* x, int64_t n, int32_t nperseg, float shift, int32_t use_abs, int32_t batch,
                 void* workspace, int64_t workspace_bytes, double* acc, int64_t* nseg_out, void* stream);

/* One segment of arbitrary length n (2 <= n <= 2^21): the reference passes nperseg = len(data) whenever the
 * window is shorter than 2^20 samples or than the requested PSD length (plot-trace.py:433-437), i.e. ONE periodic-
 * Hann segment that is not a power of two.  Bluestein chirp-z on the same register-resident FFT.  `mean` = the
 * segment mean the caller computed (float64; of |x| if use_abs); acc[k] = |rfft(w (x - mean))[k]|^2, k = 0..n/2.   */
int64_t ct_welch_single_workspace_bytes(int64_t n);
int ct_welch_single_f32(const float* x, int64_t n, double mean, int32_t use_abs, void* workspace, int64_t workspace_bytes,
                        double* acc, void* stream);

/* ---- loaders: the byte formats either side of the path ---------------------------
 * ".bin" records (>f8 curr_pA, >f8 volt_mV), print_trace.py:33-34 / noise-fit.py:90-91:
 * n records of 16 bytes -> float32 current.  Legacy (>i2, >i2) records times savegain,
 * legacy/minimal_psd.py:188-193.  ct_dequant_u16 is plot-trace.py:272-287 alone (float64
 * affine, rounded once), for series whose files have different gains.  ct_radix_hist_f32 is
 * one 8-bit digit pass (most significant first) of an exact radix select over the
 * order-preserving uint32 keys of the floats (hist256: uint64[256], caller-zeroed): the
 * median np.pad(mode='median') needs for float input.                                    */
int ct_bin_be_f64_to_f32(const void* records, int64_t n, float* out, void* stream);
int ct_i2be_to_f32(const void* records, int64_t n, float gain, float* out, void* stream);
int ct_dequant_u16(const uint16_t* raw, int64_t n, uint16_t mask, double alpha, double beta, float* out,
                   void* stream);
int ct_radix_hist_f32(const float* x, int64_t n, uint32_t prefix, int32_t prefix_bits, int32_t use_abs,
                      uint64_t* hist256, void* stream);

#ifdef __cplusplus
}
#endif
#endif
