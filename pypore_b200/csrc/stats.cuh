// stats.cuh -- K4: Segment.mean / std / min / max (PyPore/core.py:209-223) as a
// segmented reduction over flat event space, fp64.
//
// A group of G lanes (8 for short rows, 32 for long ones) owns one row (segment or event).
// std is computed from deviations, never from prefix-sum differences (SURVEY App. D.3):
//   * rows of at most K4_ONE_PASS samples: ONE pass with the shift K = the row's first sample:
//     d = x - K,  m1 = sum(d)/n,  mean = K + m1,  var = sum(d*d)/n - m1^2.  Each lane adds k = n/G terms
//     and the group adds its G lane sums, so with u = 2^-53 the sums carry errors up to
//     (k + log2 G) u sum|d| and (k + log2 G) u sum(d*d) (sum(d*d) = n (var + m1^2)).  Hence
//       |error of mean| <~ (k + log2 G + 2) u (|m1| + sqrt(var))   (mean|d| <= |m1| + sqrt(var)),
//       relative error of var <~ (k + log2 G + 3) u (1 + m1^2 / var).
//     Both grow with m1^2 / var = (K - mean)^2 / var, which reaches n when K is the row's worst outlier:
//     at n = 65536 the first-order bounds are ~1e-6 and the errors were measured at several 1e-9 (one
//     float32 sample of 1000.123 followed by 65,535 samples of 1e-3).  So a row with m1^2 > 2^10 var is
//     summed again in two passes (next point); below that the var bound is 1025 (k + 8) u < 1e-9 and the
//     mean error < 33 (k + 7) u sqrt(var), no more than the two-pass sum's own (k + 5) u mean|x| allows
//     for a row whose spread is not tiny against its mean.  Constant rows come out exact (d = 0);
//   * samples travel as 16-byte vectors (float4 / double2) from the row's 16-byte-aligned start, the
//     elements in front of and behind the row are masked: a row of ~130 float32 samples is 5 trips of an
//     8-lane group instead of 17 (the first cut issued 32 thread instructions per sample, most of them
//     per-row set-up and scalar loads: 31 % of the HBM peak);
//   * longer rows and the rows above: two passes (mean = sum(x)/n, then
//     the deviations from it), like np.std, from scalar loads; a finite constant row gets its value and 0.
// min / max run on the samples' own type (int16 ADC counts: on the counts, decoded at the end); a NaN anywhere
// makes both NaN like np.min / np.max.
#pragma once
#include "common.cuh"

constexpr int K4_ONE_PASS = 65536;
constexpr int K4_U = 4;  // independent 16-byte loads per lane and trip (8 lanes x 4 x float4 = 128 samples: most rows are one trip)

template <int G>
__device__ __forceinline__ double k4_group_sum(double v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v += __shfl_xor_sync(PP_FULL, v, d);
    return v;
}
template <int G>
__device__ __forceinline__ float k4_group_min(float v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = fminf(v, __shfl_xor_sync(PP_FULL, v, d));
    return v;
}
template <int G>
__device__ __forceinline__ float k4_group_max(float v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(PP_FULL, v, d));
    return v;
}
template <int G>
__device__ __forceinline__ double k4_group_min(double v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = fmin(v, __shfl_xor_sync(PP_FULL, v, d));
    return v;
}
template <int G>
__device__ __forceinline__ double k4_group_max(double v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(PP_FULL, v, d));
    return v;
}
template <int G>
__device__ __forceinline__ int16_t k4_group_min(int16_t v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = min(v, (int16_t)__shfl_xor_sync(PP_FULL, (int)v, d));
    return v;
}
template <int G>
__device__ __forceinline__ int16_t k4_group_max(int16_t v)
{
#pragma unroll
    for (int d = G / 2; d > 0; d >>= 1) v = max(v, (int16_t)__shfl_xor_sync(PP_FULL, (int)v, d));
    return v;
}
__device__ __forceinline__ float k4_min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float k4_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double k4_min(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ double k4_max(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ int16_t k4_min(int16_t a, int16_t b) { return a < b ? a : b; }
__device__ __forceinline__ int16_t k4_max(int16_t a, int16_t b) { return a > b ? a : b; }

template <typename T> struct K4Vec;
template <> struct K4Vec<float> {
    static constexpr int N = 4;
    typedef float4 V;
    static __device__ __forceinline__ void get(const V &q, float *o) { o[0] = q.x; o[1] = q.y; o[2] = q.z; o[3] = q.w; }
};
template <> struct K4Vec<double> {
    static constexpr int N = 2;
    typedef double2 V;
    static __device__ __forceinline__ void get(const V &q, double *o) { o[0] = q.x; o[1] = q.y; }
};
template <> struct K4Vec<int16_t> {   // ADC counts: min / max on the counts, decoded once at the end
    static constexpr int N = 8;
    typedef int4 V;
    static __device__ __forceinline__ void get(const V &q, int16_t *o)
    {
        const int w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { o[2 * i] = (int16_t)(w[i] & 0xffff); o[2 * i + 1] = (int16_t)(w[i] >> 16); }
    }
};
// start values of the min / max tracking: +-inf, or the ends of the int16 range
template <typename T> __device__ __forceinline__ T k4_top() { return (T)__longlong_as_double(0x7ff0000000000000LL); }
template <> __device__ __forceinline__ int16_t k4_top<int16_t>() { return 32767; }
template <typename T> __device__ __forceinline__ T k4_bottom() { return -k4_top<T>(); }
template <> __device__ __forceinline__ int16_t k4_bottom<int16_t>() { return -32768; }

// Rows k = group, group + ngroups, ...; every lane of a warp runs the same number of rows
// so that the full-mask shuffles stay convergent (inactive groups work on an empty row).
template <typename T, int G>
__device__ __forceinline__ void k4_rows(const T *__restrict__ samples, const int64_t *__restrict__ ev_base,
                                        const int64_t *__restrict__ ev_off, int64_t row0, int64_t rows, int64_t total,
                                        const int64_t *__restrict__ flat_start, const int *__restrict__ row_event,
                                        double *__restrict__ o_mean, double *__restrict__ o_std,
                                        double *__restrict__ o_min, double *__restrict__ o_max, const PPAdc &adc)
{
    typedef K4Vec<T> VT;
    constexpr int N = VT::N;
    const int gl = threadIdx.x & (G - 1);
    const int64_t group0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngroups = ((int64_t)gridDim.x * blockDim.x) / G;
    const int64_t warp_first = group0 - ((threadIdx.x & 31) / G);  // row of the warp's first group
    for (int64_t kw = row0 + warp_first; kw < rows; kw += ngroups) {  // rows [row0, rows)
        const int64_t k = kw + ((threadIdx.x & 31) / G);
        const bool live = k < rows;
        int64_t len = 0;
        const T *p = samples;
        if (live) {
            const int64_t f0 = flat_start[k];
            const int64_t f1 = (k + 1 < rows) ? flat_start[k + 1] : total;
            const int64_t ev = row_event ? (int64_t)row_event[k] : k;
            len = f1 - f0;
            p = samples + ev_base[ev] + (f0 - ev_off[ev]);
        }
        double s1 = 0.0, s2 = 0.0;
        T mn = k4_top<T>(), mx = k4_bottom<T>();
        int nan = 0;
        double mean, var;
        // Which passes a row takes depends on the row alone, never on the rows that share its warp: the streamed
        // pipeline's per-chunk launches start at another row (seg_done) than one launch over the whole table, and
        // both must give the same bits.  A long row's group runs the one-pass loop over nothing, the two-pass
        // block below over its row (shuffles stay warp-wide in both).
        const bool long_row = len > K4_ONE_PASS;
        const int64_t n1 = long_row ? 0 : len;
        bool redo = long_row;  // this group's row takes the two passes
        if (__any_sync(PP_FULL, !long_row)) {
            // 16-byte vectors from the aligned start: `mis` elements of the first vector lie in front of the row
            const int mis = (int)((reinterpret_cast<uintptr_t>(p) & 15) / sizeof(T));
            const typename VT::V *pv = reinterpret_cast<const typename VT::V *>(p - mis);
            const int64_t last = mis + n1;                   // elements [mis, last) of the vector stream are the row
            const int64_t nvec = (last + N - 1) / N;
            double K = n1 > 0 ? pp_val(__ldg(p), adc) : 0.0;  // the shift: the row's first sample
            if (!(fabs(K) <= 1.7e308)) K = 0.0;              // inf / NaN: plain sums
            for (int64_t v0 = gl; v0 < nvec; v0 += K4_U * G) {
                typename VT::V q[K4_U];
#pragma unroll
                for (int u = 0; u < K4_U; ++u)
                    if (v0 + u * G < nvec) q[u] = __ldg(pv + v0 + u * G);
#pragma unroll
                for (int u = 0; u < K4_U; ++u) {
                    const int64_t e0 = (v0 + u * G) * N;
                    if (v0 + u * G >= nvec) continue;
                    T x[N];
                    VT::get(q[u], x);
                    if (e0 >= mis && e0 + N <= last) {
#pragma unroll
                        for (int c = 0; c < N; ++c) {
                            const double d = pp_val(x[c], adc) - K;
                            s1 += d;
                            s2 = fma(d, d, s2);
                            mn = k4_min(mn, x[c]);
                            mx = k4_max(mx, x[c]);
                            nan |= (x[c] != x[c]);
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < N; ++c) {
                            if (e0 + c >= mis && e0 + c < last) {
                                const double d = pp_val(x[c], adc) - K;
                                s1 += d;
                                s2 = fma(d, d, s2);
                                mn = k4_min(mn, x[c]);
                                mx = k4_max(mx, x[c]);
                                nan |= (x[c] != x[c]);
                            }
                        }
                    }
                }
            }
            s1 = k4_group_sum<G>(s1);
            s2 = k4_group_sum<G>(s2);
            const double rl = 1.0 / (double)(n1 > 0 ? n1 : 1);
            const double m1 = s1 * rl;
            mean = K + m1;
            var = s2 * rl - m1 * m1;
            if (n1 == 0) { mean = __longlong_as_double(0x7ff8000000000000LL); var = mean; }
            // heavy cancellation: the shift sits far from the mean (false for NaN)
            redo = long_row || m1 * m1 > 1024.0 * var;
        }
        if (__any_sync(PP_FULL, redo)) {
            // rows of the other groups run with length 0: the group sums below are warp-wide
            const int64_t n2 = redo ? len : 0;
            double t1 = 0.0, t2 = 0.0;
            for (int64_t j = gl; j < n2; j += G) {
                const T x = p[j];
                t1 += pp_val(x, adc);
                if (long_row) {
                    mn = k4_min(mn, x);
                    mx = k4_max(mx, x);
                    nan |= (x != x);
                }
            }
            const double m2 = k4_group_sum<G>(t1) / (double)len;
            for (int64_t j = gl; j < n2; j += G) {
                const double d = pp_val(p[j], adc) - m2;
                t2 = fma(d, d, t2);
            }
            t2 = k4_group_sum<G>(t2);
            if (redo) { mean = m2; var = t2 / (double)len; }
        }
        mn = k4_group_min<G>(mn);
        mx = k4_group_max<G>(mx);
#pragma unroll
        for (int d = G / 2; d > 0; d >>= 1) nan |= __shfl_xor_sync(PP_FULL, nan, d);
        if (long_row && !nan && mn == mx) {  // a finite constant row: its value and exactly 0, as in one pass
            const double v = pp_val(mn, adc);
            if (fabs(v) <= 1.7e308) { mean = v; var = 0.0; }
        }
        if (live && gl == 0) {
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            double dmn = pp_val(mn, adc), dmx = pp_val(mx, adc);
            if (sizeof(T) == 2 && adc.scale < 0.0) { const double t = dmn; dmn = dmx; dmx = t; }  // decreasing decode
            o_mean[k] = mean;
            o_std[k] = sqrt(var < 0.0 ? 0.0 : var);
            o_min[k] = nan ? qnan : dmn;
            o_max[k] = nan ? qnan : dmx;
        }
    }
}

// flat_start[k] .. flat_start[k+1] (or `total` for the last) bounds row k;
// row_event == nullptr means row k is event k (statistics of whole events).  `adc` decodes int16 samples.
template <typename T>
__global__ void __launch_bounds__(256)
k4_segment_stats(const T *__restrict__ samples, const int64_t *__restrict__ ev_base,
                 const int64_t *__restrict__ ev_off, const PPCounters *ctr, int rows_are_events,
                 const int64_t *__restrict__ flat_start, const int *__restrict__ row_event,
                 int64_t cap_rows, double *__restrict__ o_mean, double *__restrict__ o_std,
                 double *__restrict__ o_min, double *__restrict__ o_max, PPAdc adc)
{
    int64_t rows = rows_are_events ? (int64_t)ctr->n_events : (int64_t)ctr->n_segments;
    if (rows > cap_rows) rows = cap_rows;
    const int64_t total = (int64_t)ctr->n_event_samples;
    // segments: only the rows not finalised yet (the whole table unless the streamed pipeline exports per chunk)
    const int64_t row0 = rows_are_events ? 0 : (int64_t)ctr->seg_done;
    if (rows <= row0) return;
    if (total / rows < 512)
        k4_rows<T, 8>(samples, ev_base, ev_off, row0, rows, total, flat_start, row_event, o_mean, o_std, o_min, o_max, adc);
    else
        k4_rows<T, 32>(samples, ev_base, ev_off, row0, rows, total, flat_start, row_event, o_mean, o_std, o_min, o_max, adc);
}
