// filter.cuh -- K5: Event.filter (PyPore/DataTypes.py:258-274), i.e.
// scipy.signal.filtfilt(b, a, x) with its defaults (odd padding of
// 3*max(len(a),len(b)) samples, lfilter_zi initial state, direct-form-II-
// transposed lfilter forward, then backward), as a parallel linear-recurrence scan.
//
// The DF2T state update is affine in the state:   z' = M z + c x,   y = z0 + b0 x
// with M[k][0] = -a[k+1], M[k][k+1] = 1.  One CTA walks one event in tiles of
// 4096 samples.  Inside a tile every thread runs the recurrence over its 16
// samples from a zero state (thread 0: from the carried state), the per-thread
// end states are combined with a Hillis-Steele scan that uses the precomputed
// powers (M^16)^(2^k), and every thread re-runs its samples from its true
// initial state.  Tiles are staged through shared memory so that global
// traffic is coalesced: 4 or 8 B read and 8 B written per sample per pass.
// Results differ from scipy's strictly sequential evaluation only by fp64
// rounding of the state propagation (tolerance in BASELINE.json: 1e-5 relative).
#pragma once
#include "common.cuh"

constexpr int FILT_MAX_COEF = 9;  // filter order <= 8
constexpr int FILT_NZ = FILT_MAX_COEF - 1;
constexpr int K5_THREADS = 256;
constexpr int K5_CH = 16;
constexpr int K5_TILE = K5_THREADS * K5_CH;  // 4096
constexpr int K5_LOG = 8;                    // log2(K5_THREADS)

struct K5Coef {
    double b[FILT_MAX_COEF], a[FILT_MAX_COEF], zi[FILT_NZ];
    double pw[K5_LOG][FILT_NZ][FILT_NZ];  // (M^K5_CH)^(2^k)
    int nc;                               // number of coefficients (order + 1)
};

template <int NZ>
__device__ __forceinline__ double k5_step(const K5Coef &C, double (&z)[NZ], double x)
{
    const double y = C.b[0] * x + z[0];
#pragma unroll
    for (int k = 0; k < NZ - 1; ++k) z[k] = C.b[k + 1] * x + z[k + 1] - C.a[k + 1] * y;
    z[NZ - 1] = C.b[NZ] * x - C.a[NZ] * y;
    return y;
}

// Sample j of the odd-extended event (scipy odd_ext), j in [0, L + 2P).
__device__ __forceinline__ double k5_ext(const PPSource &src, int64_t ev, int64_t L, int P, int64_t j)
{
    if (j < P) return 2.0 * pp_sample(src, ev, 0) - pp_sample(src, ev, P - j);
    if (j < P + L) return pp_sample(src, ev, j - P);
    return 2.0 * pp_sample(src, ev, L - 1) - pp_sample(src, ev, L - 2 - (j - P - L));
}

// One direction of filtfilt for every event.
//   backward == 0: input = odd extension of the event, output tmp[toff + j]
//   backward == 1: input = tmp reversed, output out[ev_off + i] (padding stripped, order restored)
template <int NZ>
__global__ void __launch_bounds__(K5_THREADS)
k5_filter_pass(PPSource src, const int64_t *__restrict__ ev_len, PPCounters *ctr,
               const K5Coef *__restrict__ coef, double *__restrict__ tmp, double *__restrict__ out,
               int backward)
{
    extern __shared__ __align__(16) unsigned char k5_smem[];
    double *tile = reinterpret_cast<double *>(k5_smem);                                 // [K5_THREADS][K5_CH + 1]
    double(*zs)[K5_THREADS][NZ] =
        reinterpret_cast<double(*)[K5_THREADS][NZ]>(tile + K5_THREADS * (K5_CH + 1));   // [2][K5_THREADS][NZ]
    double *carry = reinterpret_cast<double *>(zs + 2);                                 // [NZ]
    K5Coef &C = *reinterpret_cast<K5Coef *>(carry + FILT_NZ);
    const int tid = threadIdx.x;
    for (int k = tid; k < (int)(sizeof(K5Coef) / sizeof(double)); k += K5_THREADS)
        reinterpret_cast<double *>(&C)[k] = reinterpret_cast<const double *>(coef)[k];
    if (tid == 0) C.nc = coef->nc;
    __syncthreads();
    const int P = 3 * (NZ + 1);
    const int64_t n_events = (int64_t)ctr->n_events;
    for (int64_t ev = blockIdx.x; ev < n_events; ev += gridDim.x) {
        const int64_t L = ev_len[ev];
        if (L <= P) {
            if (tid == 0) atomicOr(&ctr->overflow, (unsigned)PP_OVF_FILTER_SHORT);
            continue;
        }
        const int64_t M = L + 2 * P;
        const int64_t off = src.ev_off[ev];
        const int64_t toff = off + 2LL * P * ev;
        __syncthreads();
        if (tid < NZ) {
            const double x0 = backward ? tmp[toff + M - 1] : k5_ext(src, ev, L, P, 0);
            carry[tid] = C.zi[tid] * x0;
        }
        for (int64_t t0 = 0; t0 < M; t0 += K5_TILE) {
            __syncthreads();
            // coalesced load of the tile into padded shared memory
            for (int q = tid; q < K5_TILE; q += K5_THREADS) {
                const int64_t j = t0 + q;
                double v = 0.0;
                if (j < M) v = backward ? tmp[toff + (M - 1 - j)] : k5_ext(src, ev, L, P, j);
                tile[(q / K5_CH) * (K5_CH + 1) + (q % K5_CH)] = v;
            }
            __syncthreads();
            // pass 1: end state of my chunk from a zero state (thread 0: from the carry)
            double z[NZ];
#pragma unroll
            for (int k = 0; k < NZ; ++k) z[k] = tid == 0 ? carry[k] : 0.0;
            double *row = tile + tid * (K5_CH + 1);
#pragma unroll
            for (int k = 0; k < K5_CH; ++k) k5_step<NZ>(C, z, row[k]);
#pragma unroll
            for (int k = 0; k < NZ; ++k) zs[0][tid][k] = z[k];
            __syncthreads();
            // inclusive scan of affine maps with a constant linear part
            int cur = 0;
#pragma unroll
            for (int s = 0; s < K5_LOG; ++s) {
                const int d = 1 << s;
                double v[NZ];
#pragma unroll
                for (int k = 0; k < NZ; ++k) v[k] = zs[cur][tid][k];
                if (tid >= d) {
#pragma unroll
                    for (int r = 0; r < NZ; ++r) {
                        double acc = v[r];
#pragma unroll
                        for (int c = 0; c < NZ; ++c) acc += C.pw[s][r][c] * zs[cur][tid - d][c];
                        v[r] = acc;
                    }
                }
#pragma unroll
                for (int k = 0; k < NZ; ++k) zs[cur ^ 1][tid][k] = v[k];
                cur ^= 1;
                __syncthreads();
            }
            // pass 2: re-run from the true initial state, in place
#pragma unroll
            for (int k = 0; k < NZ; ++k) z[k] = tid == 0 ? carry[k] : zs[cur][tid - 1][k];
#pragma unroll
            for (int k = 0; k < K5_CH; ++k) row[k] = k5_step<NZ>(C, z, row[k]);
            __syncthreads();
            if (tid < NZ) carry[tid] = zs[cur][K5_THREADS - 1][tid];
            // coalesced store
            for (int q = tid; q < K5_TILE; q += K5_THREADS) {
                const int64_t j = t0 + q;
                if (j >= M) break;
                const double v = tile[(q / K5_CH) * (K5_CH + 1) + (q % K5_CH)];
                if (!backward) tmp[toff + j] = v;
                else {
                    const int64_t p = M - 1 - j;  // position in the extended signal
                    if (p >= P && p < P + L) out[off + (p - P)] = v;
                }
            }
        }
    }
}

// Orders >= 3: the DF2T state space is too badly scaled for matrix-power propagation
// (measured: 2.4e-4 of max|y| at order 3 and fc/fs = 1e-3, 2e-8 relative error at order 4, 4e-2 at
// order 6), so those run in scipy's own strictly sequential operation order, one thread per event and
// direction.  Orders 1 and 2 stay within 1.3e-10 of max|y| for fc/fs in [1e-3, 0.2] up to 4 M samples.
template <int NZ>
__global__ void __launch_bounds__(64)
k5_filter_sequential(PPSource src, const int64_t *__restrict__ ev_len, PPCounters *ctr,
                     const K5Coef *__restrict__ coef, double *__restrict__ tmp, double *__restrict__ out,
                     int backward)
{
    __shared__ K5Coef C;
    for (int k = threadIdx.x; k < (int)(sizeof(K5Coef) / sizeof(double)); k += blockDim.x)
        reinterpret_cast<double *>(&C)[k] = reinterpret_cast<const double *>(coef)[k];
    __syncthreads();
    const int P = 3 * (NZ + 1);
    const int64_t n_events = (int64_t)ctr->n_events;
    for (int64_t ev = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; ev < n_events;
         ev += (int64_t)gridDim.x * blockDim.x) {
        const int64_t L = ev_len[ev];
        if (L <= P) { atomicOr(&ctr->overflow, (unsigned)PP_OVF_FILTER_SHORT); continue; }
        const int64_t M = L + 2 * P;
        const int64_t off = src.ev_off[ev];
        const int64_t toff = off + 2LL * P * ev;
        double z[NZ];
        const double x0 = backward ? tmp[toff + M - 1] : k5_ext(src, ev, L, P, 0);
#pragma unroll
        for (int k = 0; k < NZ; ++k) z[k] = C.zi[k] * x0;
        for (int64_t j = 0; j < M; ++j) {
            const double x = backward ? tmp[toff + (M - 1 - j)] : k5_ext(src, ev, L, P, j);
            const double y = k5_step<NZ>(C, z, x);
            if (!backward) tmp[toff + j] = y;
            else {
                const int64_t p = M - 1 - j;
                if (p >= P && p < P + L) out[off + (p - P)] = y;
            }
        }
    }
}

template <int NZ>
constexpr size_t k5_smem_bytes()
{
    return sizeof(double) * (K5_THREADS * (K5_CH + 1) + 2 * K5_THREADS * NZ + FILT_NZ) + sizeof(K5Coef);
}

// Host side: powers of the state-transition matrix (tiny; done per call).
static void k5_prepare(const double *b, const double *a, const double *zi, int nc, K5Coef *C)
{
    memset(C, 0, sizeof *C);
    const int nz = nc - 1;
    for (int i = 0; i < nc; ++i) { C->b[i] = b[i]; C->a[i] = a[i]; }
    for (int i = 0; i < nz; ++i) C->zi[i] = zi[i];
    C->nc = nc;
    double Mx[FILT_NZ][FILT_NZ] = {{0}}, R[FILT_NZ][FILT_NZ], Tm[FILT_NZ][FILT_NZ];
    for (int k = 0; k < nz; ++k) {
        Mx[k][0] = -a[k + 1];
        if (k + 1 < nz) Mx[k][k + 1] += 1.0;
    }
    // R = M^K5_CH by repeated multiplication
    for (int r = 0; r < nz; ++r)
        for (int c = 0; c < nz; ++c) R[r][c] = (r == c) ? 1.0 : 0.0;
    for (int it = 0; it < K5_CH; ++it) {
        for (int r = 0; r < nz; ++r)
            for (int c = 0; c < nz; ++c) {
                double s = 0.0;
                for (int k = 0; k < nz; ++k) s += Mx[r][k] * R[k][c];
                Tm[r][c] = s;
            }
        memcpy(R, Tm, sizeof R);
    }
    for (int s = 0; s < K5_LOG; ++s) {
        for (int r = 0; r < nz; ++r)
            for (int c = 0; c < nz; ++c) C->pw[s][r][c] = R[r][c];
        for (int r = 0; r < nz; ++r)
            for (int c = 0; c < nz; ++c) {
                double sum = 0.0;
                for (int k = 0; k < nz; ++k) sum += R[r][k] * R[k][c];
                Tm[r][c] = sum;
            }
        memcpy(R, Tm, sizeof R);
    }
}
