// common.cuh -- shared declarations for the sm_100a segmentation kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/pypore_b200.h"

#define PP_WARP 32
#define PP_FULL 0xffffffffu

// Device-side counters, one instance per context (zeroed per stage as needed).
struct PPCounters {
    unsigned long long n_edges[2];    // K1 threshold crossings found so far (two slots: k1_stitch reads one, writes the other)
    unsigned long long n_runs;        // n_edges + 1 (0 for an empty trace)
    unsigned long long n_events;
    unsigned long long n_event_samples;
    unsigned long long n_segments;
    // split work queue
    unsigned long long q_head;        // next ticket to consume
    unsigned long long q_tail;        // next slot to fill
    long long q_pending;              // tasks pushed and not yet finished
    unsigned long long n_cand;        // candidate evaluations
    unsigned long long n_scan;        // window scans
    unsigned long long n_tasks;       // tasks processed
    unsigned long long n_exact;       // exact (reference-arithmetic) candidate evaluations
    unsigned long long n_sure;        // screened windows decided on the screened gain alone
    unsigned long long n_multi;       // screened windows decided by the argmax over several contenders' exact gains
    unsigned long long n_full;        // windows scanned exactly in full although screening was on
    unsigned long long n_seq_redo;    // events whose prefix sums were redone sequentially
    unsigned long long n_scan_tiles;  // prefix-scan tiles over all events
    // incremental (streamed) pipeline: the stages after the threshold scan work on the events
    // [ev_begin, n_events) and the prefix-scan tiles [tile_begin, n_scan_tiles) added by the last select
    unsigned long long sel_next_run;  // first run the next incremental select looks at
    unsigned long long ev_begin;
    unsigned long long tile_begin;
    unsigned long long n_long;        // events of the current search that k3_spine walks first
    // tables finalised so far (streamed pipeline with host export: compaction, statistics and the copy-out run per
    // chunk on the flat range [flat_done, n_event_samples) / the events [ev_done, n_events)); all zero otherwise
    unsigned long long seg_done;
    unsigned long long flat_done;
    unsigned long long ev_done;
    unsigned int overflow;            // bit0 runs, bit1 queue, bit2 segments, bit3 filter-too-short
    unsigned int first_below;         // below-threshold bit of sample 0
};

enum { PP_OVF_RUNS = 1, PP_OVF_QUEUE = 2, PP_OVF_SEGS = 4, PP_OVF_FILTER_SHORT = 8,
       PP_OVF_HALO = 16 /* multi-GPU: the speculative halo did not cover a straddling event */,
       PP_OVF_EXPORT = 32 /* host tables of pp_pipeline_host_tables too small */,
       PP_OVF_CTL = 64 /* multi-GPU: a peer's record did not arrive (pp_ctl_exchange timed out) */ };

// int16 ADC counts and what they stand for: current = fl(fl(c * scale) + offset), two IEEE roundings and no FMA --
// exactly what NumPy computes for counts.astype(np.float64) * scale + offset.
struct PPAdc {
    double scale, offset;
};
__device__ __forceinline__ double pp_adc_decode(int c, const PPAdc &a)
{
    return __dadd_rn(__dmul_rn((double)c, a.scale), a.offset);
}
// A sample as the float64 value every stage computes with (float32 / float64 samples as they are)
__device__ __forceinline__ double pp_val(float x, const PPAdc &) { return (double)x; }
__device__ __forceinline__ double pp_val(double x, const PPAdc &) { return x; }
__device__ __forceinline__ double pp_val(int16_t c, const PPAdc &a) { return pp_adc_decode(c, a); }

// Where an event's samples live.
//   kind 0: float32 trace, sample j of event e = trace[ev_start[e] + j]
//   kind 1: float64 packed array, sample j of event e = flat[ev_off[e] + j]   (uploaded events, filtered current)
//   kind 2: float64 trace, sample j of event e = trace64[ev_start[e] + j]
//   kind 3: int16 ADC trace, sample j of event e = decode(trace16[ev_start[e] + j]) with `adc`
struct PPSource {
    const float *trace;
    const double *trace64;
    const int16_t *trace16;
    const double *flat;
    const int64_t *ev_start;
    const int64_t *ev_off;
    PPAdc adc;
    int kind;
};
enum { PP_SRC_TRACE32 = 0, PP_SRC_FLAT64 = 1, PP_SRC_TRACE64 = 2, PP_SRC_ADC16 = 3 };

__device__ __forceinline__ double pp_sample(const PPSource &s, int64_t ev, int64_t j)
{
    if (s.kind == PP_SRC_TRACE32) return (double)__ldg(s.trace + s.ev_start[ev] + j);
    if (s.kind == PP_SRC_TRACE64) return __ldg(s.trace64 + s.ev_start[ev] + j);
    if (s.kind == PP_SRC_ADC16) return pp_adc_decode(__ldg(s.trace16 + s.ev_start[ev] + j), s.adc);
    return __ldg(s.flat + s.ev_off[ev] + j);
}

// Monotone float32 -> uint32 key (larger float <=> larger key; -0.0 < +0.0).
__device__ __forceinline__ unsigned pp_fkey(float x)
{
    unsigned b = __float_as_uint(x);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float pp_fkey_inv(unsigned k)
{
    unsigned b = k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu);
    return __uint_as_float(b);
}
// Min tracking: NaN -> 0 (dominates the min like np.min), empty = 0xffffffff.
// Max tracking: NaN -> 0xffffffff (dominates the max like np.max), empty = 0.
#define PP_MINKEY_EMPTY 0xffffffffu
#define PP_MAXKEY_EMPTY 0u

__device__ __forceinline__ double pp_decode_min(unsigned k)
{
    if (k == 0u || k == PP_MINKEY_EMPTY) return __longlong_as_double(0x7ff8000000000000LL);
    return (double)pp_fkey_inv(k);
}
__device__ __forceinline__ double pp_decode_max(unsigned k)
{
    if (k == 0xffffffffu || k == PP_MAXKEY_EMPTY) return __longlong_as_double(0x7ff8000000000000LL);
    return (double)pp_fkey_inv(k);
}

// Largest index i in [0, n) with a[i] <= v, for a sorted ascending with a[0] <= v.
__device__ __forceinline__ int64_t pp_upper_index(const int64_t *a, int64_t n, int64_t v)
{
    int64_t lo = 0, hi = n;  // invariant: a[lo] <= v, (hi == n or a[hi] > v)
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ unsigned long long pp_ld_volatile_u64(const unsigned long long *p)
{
    return *((const volatile unsigned long long *)p);
}
