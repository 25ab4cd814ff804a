// hmm.cuh -- hidden Markov model decoding of sequences of segment means (the step PyPore feeds its segment tables
// to: Event.apply_hmm / the HMM branch of Event.parse, reference DataTypes.py:292-355).
//
// Model: S <= 128 emitting states with normal emissions, staged once per CTA in shared memory as one block of
// doubles [mu | r = 1/sigma | c = -log(sigma) - log(2 pi)/2 | log pi | log end | log A (S x S, [i*S + j])].  Every
// log is taken by the host; Viterbi evaluates no transcendental function on the device.
//
// Emission e_j(x) = c_j - 0.5 * (z * z), z = (x - mu_j) * r_j: one IEEE rounding per operation, no FMA, in NumPy's
// order -- bit-equal to NumPy's elementwise result.  Viterbi: delta_t(j) = max_i fl(delta_{t-1}(i) + logA_ij) +
// e_j(x_t), i ascending with strict >, so ties go to the lowest predecessor; logp = max_j fl(delta_T(j) + logend_j),
// lowest j on ties.  A NaN sample makes logp NaN, an impossible sequence makes it -inf; both leave every state -1.
// Forward: the same recursion with max replaced by m + log(sum_i exp(v_i - m)) (-inf when m is -inf).
//
// Layout: S <= 32: one warp per sequence, lane = state, delta broadcast with __shfl_sync; 32 < S <= 128: one CTA of
// 128 threads per sequence, delta double-buffered in shared memory, one barrier per step.  The threads of one
// predecessor i read logA[i*S .. i*S + S), consecutive words.  Persistent CTAs take sequences from an atomic counter.
// Viterbi writes one uint8 backpointer per (sample, state); k_hmm_traceback then walks each sequence back from its
// last state, one thread per sequence: a chain of T dependent loads.
#pragma once
#include "common.cuh"

constexpr int HMM_MAX_STATES = 128;
constexpr int HMM_WARP_THREADS = 256;  // 8 sequences in flight per CTA of the warp kernel
constexpr int HMM_CTA_THREADS = 128;   // one thread per state

__host__ __device__ __forceinline__ size_t hmm_model_words(int S) { return 5 * (size_t)S + (size_t)S * S; }

// The sequences of one decode: sequence k is x[off[k] .. off[k+1]), every one at least one sample long.
struct HMMSeqs {
    const double *x;
    const int64_t *off;
    int64_t n;
    double *logp;                // [n]
    int *state;                  // [off[n]] (Viterbi)
    unsigned char *bp;           // [off[n] * S] (Viterbi): bp[(off[k] + t) * S + j] = predecessor of j at step t
    unsigned long long *next;    // work counter, zero at launch
};

__device__ __forceinline__ double hmm_emit(double x, double mu, double r, double c)
{
    const double z = __dmul_rn(__dsub_rn(x, mu), r);
    return __dsub_rn(c, __dmul_rn(0.5, __dmul_rn(z, z)));
}

__device__ __forceinline__ void hmm_stage_model(double *sm, const double *__restrict__ model, int S)
{
    const size_t W = hmm_model_words(S);
    for (size_t i = threadIdx.x; i < W; i += blockDim.x) sm[i] = model[i];
    __syncthreads();
}

// (value, index) pairs: the larger value wins, the lower index on equal values
__device__ __forceinline__ void hmm_take_max(double &v, int &j, double ov, int oj)
{
    if (ov > v || (ov == v && oj < j)) { v = ov; j = oj; }
}

__device__ __forceinline__ void hmm_warp_argmax(double &v, int &j)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const double ov = __shfl_down_sync(PP_FULL, v, d);
        const int oj = __shfl_down_sync(PP_FULL, j, d);
        hmm_take_max(v, j, ov, oj);
    }
}

__device__ __forceinline__ double hmm_warp_max(double v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(PP_FULL, v, d));
    return v;
}

// S <= 32: lane j of a warp is state j; lanes >= S carry -inf.
template <bool VITERBI>
__global__ void __launch_bounds__(HMM_WARP_THREADS)
k_hmm_warp(const double *__restrict__ model, int S, HMMSeqs Q)
{
    extern __shared__ double hmm_sm[];
    hmm_stage_model(hmm_sm, model, S);
    const double NEG = -INFINITY;
    const int lane = threadIdx.x & 31;
    const bool on = lane < S;
    const int j = on ? lane : 0;
    const double *A = hmm_sm + 5 * S;
    const double mu = hmm_sm[j], r = hmm_sm[S + j], c = hmm_sm[2 * S + j], lpi = hmm_sm[3 * S + j],
                 lend = hmm_sm[4 * S + j];
    for (;;) {
        unsigned long long k = 0;
        if (lane == 0) k = atomicAdd(Q.next, 1ull);
        k = __shfl_sync(PP_FULL, k, 0);
        if ((int64_t)k >= Q.n) break;
        const int64_t a = Q.off[k], T = Q.off[k + 1] - a;
        const double *x = Q.x + a;
        double xt = x[0];
        bool nan = isnan(xt);
        double d = on ? __dadd_rn(lpi, hmm_emit(xt, mu, r, c)) : NEG;
        for (int64_t t = 1; t < T; ++t) {
            xt = x[t];
            nan |= isnan(xt);
            double best = __dadd_rn(__shfl_sync(PP_FULL, d, 0), A[j]);
            if (VITERBI) {
                int arg = 0;
                for (int i = 1; i < S; ++i) {
                    const double v = __dadd_rn(__shfl_sync(PP_FULL, d, i), A[i * S + j]);
                    if (v > best) { best = v; arg = i; }
                }
                if (on) Q.bp[(a + t) * S + lane] = (unsigned char)arg;
            } else {
                for (int i = 1; i < S; ++i) best = fmax(best, __dadd_rn(__shfl_sync(PP_FULL, d, i), A[i * S + j]));
                // every lane runs the shuffles (best differs per lane); a state with no finite predecessor sums zeros
                const double m = best == NEG ? 0.0 : best;
                double s = 0.0;
                for (int i = 0; i < S; ++i) s += exp(__dadd_rn(__shfl_sync(PP_FULL, d, i), A[i * S + j]) - m);
                if (best != NEG) best += log(s);
            }
            d = on ? __dadd_rn(best, hmm_emit(xt, mu, r, c)) : NEG;
        }
        double v = on ? __dadd_rn(d, lend) : NEG;
        if (VITERBI) {
            int jj = lane;
            hmm_warp_argmax(v, jj);
            if (lane == 0) {
                const bool none = nan || v == NEG;
                Q.logp[k] = nan ? __longlong_as_double(0x7ff8000000000000LL) : v;
                Q.state[a + T - 1] = none ? -1 : jj;
            }
        } else {
            const double m = hmm_warp_max(v);
            double s = 0.0;
            for (int i = 0; i < S; ++i) s += exp(__shfl_sync(PP_FULL, v, i) - (m == NEG ? 0.0 : m));
            if (lane == 0)
                Q.logp[k] = nan ? __longlong_as_double(0x7ff8000000000000LL) : (m != NEG ? m + log(s) : m);
        }
    }
}

// 32 < S <= 128: thread j of a 128-thread CTA is state j; delta double-buffered behind the model in shared memory.
template <bool VITERBI>
__global__ void __launch_bounds__(HMM_CTA_THREADS)
k_hmm_cta(const double *__restrict__ model, int S, HMMSeqs Q)
{
    extern __shared__ double hmm_sm[];
    __shared__ unsigned long long s_k;
    hmm_stage_model(hmm_sm, model, S);
    const double NEG = -INFINITY;
    const int tid = threadIdx.x;
    const bool on = tid < S;
    const int j = on ? tid : 0;
    const double *A = hmm_sm + 5 * S;
    double *dl = hmm_sm + hmm_model_words(S);   // [2][HMM_MAX_STATES]
    const double mu = hmm_sm[j], r = hmm_sm[S + j], c = hmm_sm[2 * S + j], lpi = hmm_sm[3 * S + j];
    for (;;) {
        if (tid == 0) s_k = atomicAdd(Q.next, 1ull);
        __syncthreads();
        const unsigned long long k = s_k;
        if ((int64_t)k >= Q.n) break;
        const int64_t a = Q.off[k], T = Q.off[k + 1] - a;
        const double *x = Q.x + a;
        double xt = x[0];
        bool nan = isnan(xt);
        dl[tid] = on ? __dadd_rn(lpi, hmm_emit(xt, mu, r, c)) : NEG;
        __syncthreads();
        for (int64_t t = 1; t < T; ++t) {
            xt = x[t];
            nan |= isnan(xt);
            const double *prev = dl + ((t - 1) & 1) * HMM_MAX_STATES;
            double *cur = dl + (t & 1) * HMM_MAX_STATES;
            if (on) {
                double best = __dadd_rn(prev[0], A[j]);
                if (VITERBI) {
                    int arg = 0;
                    for (int i = 1; i < S; ++i) {
                        const double v = __dadd_rn(prev[i], A[i * S + j]);
                        if (v > best) { best = v; arg = i; }
                    }
                    Q.bp[(a + t) * S + j] = (unsigned char)arg;
                } else {
                    for (int i = 1; i < S; ++i) best = fmax(best, __dadd_rn(prev[i], A[i * S + j]));
                    if (best != NEG) {
                        double s = 0.0;
                        for (int i = 0; i < S; ++i) s += exp(__dadd_rn(prev[i], A[i * S + j]) - best);
                        best += log(s);
                    }
                }
                cur[j] = __dadd_rn(best, hmm_emit(xt, mu, r, c));
            }
            __syncthreads();
        }
        // termination in warp 0: lane l holds states l, l+32, l+64, l+96 (ascending, strict >: the lowest on ties)
        if (tid < 32) {
            const double *last = dl + ((T - 1) & 1) * HMM_MAX_STATES;
            const double *lend = hmm_sm + 4 * S;
            double v = NEG;
            int jj = tid;
            for (int q = tid; q < S; q += 32) {
                const double w = __dadd_rn(last[q], lend[q]);
                if (q == tid || w > v) { v = w; jj = q; }
            }
            if (VITERBI) {
                hmm_warp_argmax(v, jj);
                if (tid == 0) {
                    const bool none = nan || v == NEG;
                    Q.logp[k] = nan ? __longlong_as_double(0x7ff8000000000000LL) : v;
                    Q.state[a + T - 1] = none ? -1 : jj;
                }
            } else {
                const double m = hmm_warp_max(v);
                double s = 0.0;
                if (m != NEG)
                    for (int q = tid; q < S; q += 32) s += exp(__dadd_rn(last[q], lend[q]) - m);
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(PP_FULL, s, d);
                if (tid == 0)
                    Q.logp[k] = nan ? __longlong_as_double(0x7ff8000000000000LL) : (m != NEG ? m + log(s) : m);
            }
        }
    }
}

// Viterbi path from the last state back: one thread per sequence, T - 1 dependent byte loads.  A sequence whose
// last state is -1 (NaN or impossible) gets -1 everywhere.
__global__ void __launch_bounds__(128)
k_hmm_traceback(HMMSeqs Q, int S)
{
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < Q.n; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = Q.off[k], b = Q.off[k + 1];
        int s = Q.state[b - 1];
        for (int64_t t = b - 1; t > a; --t) {
            if (s >= 0) s = Q.bp[t * S + s];
            Q.state[t - 1] = s;
        }
    }
}

// off[e] = first segment row of event e (seg_event is sorted), off[n_events] = n_rows
__global__ void __launch_bounds__(256)
k_hmm_event_offsets(const int *__restrict__ seg_event, int64_t n_rows, int64_t n_events, int64_t *__restrict__ off)
{
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e <= n_events;
         e += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = n_rows;   // first row with seg_event >= e
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (seg_event[mid] < e) lo = mid + 1; else hi = mid;
        }
        off[e] = lo;
    }
}

// HMM-guided merge, step 1: the breakpoint bitmap rebuilt from the segment starts that survive -- the first segment
// of an event, and every segment whose Viterbi state is -1 or differs from its predecessor's.  (The split search's
// bitmap is not kept intact by the streamed pipeline, so it is not edited in place.)
__global__ void __launch_bounds__(256)
k_hmm_merge_bits(const int *__restrict__ seg_event, const int64_t *__restrict__ seg_flat,
                 const int *__restrict__ state, int64_t n_rows, unsigned *__restrict__ bits)
{
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n_rows; k += (int64_t)gridDim.x * blockDim.x) {
        const bool keep = k == 0 || seg_event[k] != seg_event[k - 1] || state[k] < 0 || state[k] != state[k - 1];
        if (keep) {
            const int64_t f = seg_flat[k];
            atomicOr(&bits[f >> 5], 1u << (unsigned)(f & 31));
        }
    }
}

// step 3, after the compaction: a merged row's state is that of the old row starting at the same flat position
__global__ void __launch_bounds__(256)
k_hmm_merged_states(const PPCounters *ctr, const int64_t *__restrict__ seg_flat, const int64_t *__restrict__ old_flat,
                    const int *__restrict__ old_state, int64_t n_old, int *__restrict__ state)
{
    const int64_t n = (int64_t)ctr->n_segments;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = seg_flat[k];
        int64_t lo = 0, hi = n_old;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (old_flat[mid] < f) lo = mid + 1; else hi = mid;
        }
        state[k] = old_state[lo];
    }
}
