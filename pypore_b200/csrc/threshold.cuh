// threshold.cuh -- K1: lambda_event_parser.parse as one streaming pass.
//
// Replaces PyPore/parsers.py:148-155 (mask / diff / where / split) and the
// np.min / np.max second pass of _lambda_select (parsers.py:136-140 through
// core.py:215-220).  One read of the trace (4 B/sample for float32 input, 8 B/sample for float64 input, 2 B/sample
// for int16 ADC counts):
//
//   k1_scan_tiles   persistent CTAs stream 4096-sample tiles through a ring of shared-memory stages filled by
//                   1-D TMA bulk copies (cp.async.bulk + mbarrier, three tiles in flight per CTA).  Each WARP owns a
//                   512-sample span of the tile and works on its own: below-threshold bits, crossings, min / max
//                   (NaN dominates like np.min / np.max).  A span without a crossing -- 11 out of 12 on the headline
//                   workload -- costs 16 compares, a vote and two 64-bit warp minima, and writes one 24-byte record.
//                   Spans with crossings also stage up to K1_STAGE of them (position, min / max of the piece that
//                   starts there).  No inter-tile dependency, no global atomic, one CTA barrier per tile (the stage
//                   hand-back).
//   k1_stitch       one thread per span record: exclusive scan of the crossing counts (decoupled look-back over
//                   1024-record blocks -- a chain of 15 for 60 M samples, off the streaming path) gives every span
//                   its first run index; run starts are written and the min / max pieces folded into the run table.
//                   A span with more than K1_STAGE crossings (noise riding on the threshold) is walked again here,
//                   sample by sample.
//   k1_finalize_runs decodes the run table (length, side, min / max as float64).
//
// ADC counts are scanned as integer keys k = c ^ kxor (kxor = -1 for a negative scale: ~c = -c - 1 reverses the
// order), in which the decoded current fl(fl(c * scale) + offset) is non-decreasing.  So `current < threshold` is
// `k < key threshold` (pp_adc16_key_threshold), the no-crossing path is a warp integer min / max and a vote, there
// is no NaN, and the run extrema are the keys' extrema, decoded once by k1_finalize_runs.
//
// The first round's kernel did all of this in one pass with the look-back inside the streaming kernel: 28 % of the
// HBM peak, 11 barrier-stall cycles per issue (profiles/r01o_ncu_summary.csv).
#pragma once
#include "common.cuh"

constexpr int K1_THREADS = 256;
constexpr int K1_WARPS = K1_THREADS / 32;
constexpr int K1_SPAN = 512;                        // samples per warp and tile
constexpr int K1_TILE = K1_WARPS * K1_SPAN;         // 4096 samples
#ifndef K1_CFG_STAGES
#define K1_CFG_STAGES 4
#endif
constexpr int K1_STAGES = K1_CFG_STAGES;            // tiles in flight per CTA
constexpr int K1_STAGE = 8;                         // crossings staged per span; more: the span is walked again by k1_stitch

// Monotone double -> uint64 key (larger double <=> larger key; -0.0 < +0.0).
__device__ __forceinline__ unsigned long long pp_dkey(double x)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return b ^ ((b >> 63) ? ~0ull : 0x8000000000000000ull);
}
__device__ __forceinline__ double pp_dkey_inv(unsigned long long k)
{
    const unsigned long long b = k ^ ((k >> 63) ? 0x8000000000000000ull : ~0ull);
    return __longlong_as_double((long long)b);
}
// Min tracking: NaN -> 0 (dominates the min like np.min), empty = ~0.  Max tracking: NaN -> ~0, empty = 0.
#define PP_MINKEY64_EMPTY (~0ull)
#define PP_MAXKEY64_EMPTY 0ull

struct K1Record {            // one per 512-sample span
    unsigned count;          // crossings inside the span (a crossing at p: sample p is on the other side than p - 1)
    unsigned first_below;    // side of the span's first sample
    unsigned long long head_min, head_max;   // keys of the samples before the first crossing (empty keys if there are none)
};

struct K1Staged {            // crossing k < K1_STAGE of a span
    unsigned long long mn, mx;               // keys of the samples from this crossing to the next one / the span's end
    unsigned pos, pad;                       // position inside the span
};

__device__ __forceinline__ unsigned long long k1_warp_min_u64(unsigned long long k)
{
    const unsigned hi = (unsigned)(k >> 32);
    const unsigned mh = __reduce_min_sync(PP_FULL, hi);
    const unsigned lo = hi == mh ? (unsigned)k : 0xffffffffu;
    const unsigned ml = __reduce_min_sync(PP_FULL, lo);
    return ((unsigned long long)mh << 32) | ml;
}
__device__ __forceinline__ unsigned long long k1_warp_max_u64(unsigned long long k)
{
    const unsigned hi = (unsigned)(k >> 32);
    const unsigned mh = __reduce_max_sync(PP_FULL, hi);
    const unsigned lo = hi == mh ? (unsigned)k : 0u;
    const unsigned ml = __reduce_max_sync(PP_FULL, lo);
    return ((unsigned long long)mh << 32) | ml;
}

// ---- mbarrier / bulk-copy plumbing (PTX; one CTA, no cluster) --------------------------------------
__device__ __forceinline__ unsigned k1_smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void k1_mbar_init(void *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(k1_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void k1_mbar_expect(void *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(k1_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void k1_mbar_wait(void *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "K1_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra K1_WAIT_LOOP;\n"
        "}\n" ::"r"(k1_smem_addr(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void k1_bulk_load(void *dst, const void *src, unsigned bytes, void *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(k1_smem_addr(dst)), "l"(src), "r"(bytes), "r"(k1_smem_addr(bar)) : "memory");
}

template <typename T> __device__ __forceinline__ T k1_min(T a, T b);
template <> __device__ __forceinline__ float k1_min<float>(float a, float b) { return fminf(a, b); }
template <> __device__ __forceinline__ double k1_min<double>(double a, double b) { return fmin(a, b); }
template <typename T> __device__ __forceinline__ T k1_max(T a, T b);
template <> __device__ __forceinline__ float k1_max<float>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ double k1_max<double>(double a, double b) { return fmax(a, b); }
template <> __device__ __forceinline__ int k1_min<int>(int a, int b) { return min(a, b); }
template <> __device__ __forceinline__ int k1_max<int>(int a, int b) { return max(a, b); }

// What the scan compares: float32 / float64 samples as they are, int16 ADC counts as their keys c ^ kxor.
template <typename T> struct K1Key {
    typedef T V;
    static __device__ __forceinline__ V of(T x, int) { return x; }
};
template <> struct K1Key<int16_t> {
    typedef int V;
    static __device__ __forceinline__ V of(int16_t c, int kxor) { return (int)c ^ kxor; }
};

// run-key extrema of a warp (keys as in the run table: pp_dkey of the value)
__device__ __forceinline__ unsigned long long k1_warp_min_key(float m) { return k1_warp_min_u64(pp_dkey((double)m)); }
__device__ __forceinline__ unsigned long long k1_warp_max_key(float m) { return k1_warp_max_u64(pp_dkey((double)m)); }
__device__ __forceinline__ unsigned long long k1_warp_min_key(double m) { return k1_warp_min_u64(pp_dkey(m)); }
__device__ __forceinline__ unsigned long long k1_warp_max_key(double m) { return k1_warp_max_u64(pp_dkey(m)); }
__device__ __forceinline__ unsigned long long k1_warp_min_key(int m) { return pp_dkey((double)__reduce_min_sync(PP_FULL, m)); }
__device__ __forceinline__ unsigned long long k1_warp_max_key(int m) { return pp_dkey((double)__reduce_max_sync(PP_FULL, m)); }

__device__ __forceinline__ void k1_mbar_arrive(void *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(k1_smem_addr(bar)) : "memory");
}

// m = min ignoring NaN, M = max PROPAGATING NaN: `m < thr` says "a sample is below", `!(M < thr)` says "a sample is
// above" (NaN compares false, i.e. counts as above, like the reference's mask), and M != M says "there is a NaN" --
// the no-crossing path needs nothing else, in particular no per-sample compare.
__device__ __forceinline__ float k1_max_nan(float a, float b)
{
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ double k1_max_nan(double a, double b) { return (a != a || b != b) ? a + b : fmax(a, b); }
__device__ __forceinline__ int k1_max_nan(int a, int b) { return max(a, b); }

// Shared memory of k1_scan_tiles: the stages (one tile each, source and destination of the bulk copy 128-byte
// aligned -- a copy that started 16 bytes before the tile to bring the previous sample along ran at a third of
// the rate), their full / empty barriers, and per-warp scratch keys for spans with crossings.
template <typename T>
struct K1Smem {
    alignas(128) T stage[K1_STAGES][K1_TILE];
    unsigned long long full[K1_STAGES], empty[K1_STAGES];
    unsigned long long smin[K1_WARPS][K1_STAGE + 1], smax[K1_WARPS][K1_STAGE + 1];
};

constexpr int K1_CTA_THREADS = K1_THREADS + 32;   // eight consumer warps + the producer warp

// Tiles [tile_begin, tile_begin + n_tiles) of the trace prefix x[0, n).  thr: `sample < thr` <=> below
// (float32 input: the smallest float32 >= the threshold, so that the comparison equals the reference's
// double(x) < threshold for every float32 x; float64 input: the threshold itself; int16 input: the key threshold,
// compared with the keys c ^ kxor).
template <typename T>
__global__ void __launch_bounds__(K1_CTA_THREADS)
k1_scan_tiles(const T *__restrict__ x, int64_t n, typename K1Key<T>::V thr, int kxor, int64_t tile_begin,
              int64_t n_tiles, K1Record *__restrict__ rec, K1Staged *__restrict__ staged)
{
    typedef typename K1Key<T>::V V;
    extern __shared__ __align__(128) unsigned char k1_raw[];
    K1Smem<T> &S = *reinterpret_cast<K1Smem<T> *>(k1_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr unsigned TILE_BYTES = (unsigned)(K1_TILE * sizeof(T));

    if (tid == 0) {
        for (int s = 0; s < K1_STAGES; ++s) { k1_mbar_init(&S.full[s], 1); k1_mbar_init(&S.empty[s], K1_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp == K1_WARPS) {
        // ---- producer warp: keeps K1_STAGES tiles in flight.  A whole tile is one 1-D TMA bulk copy; a ragged last
        //      one is not staged at all (the consumer warps read their spans of it straight from global memory) ----
        for (int64_t it = 0; it < my_tiles; ++it) {
            const int64_t base = (tile_begin + blockIdx.x + it * (int64_t)gridDim.x) * K1_TILE;
            const int s = (int)(it % K1_STAGES);
            if (it >= K1_STAGES) k1_mbar_wait(&S.empty[s], (unsigned)((it / K1_STAGES - 1) & 1));
            if (base + K1_TILE <= n) {
                if (lane == 0) {
                    k1_mbar_expect(&S.full[s], TILE_BYTES);
                    k1_bulk_load(&S.stage[s][0], x + base, TILE_BYTES, &S.full[s]);
                }
            } else if (lane == 0) {
                k1_mbar_arrive(&S.full[s]);      // ragged last tile: nothing staged, the phase still completes
            }
        }
        return;
    }

    for (int64_t it = 0; it < my_tiles; ++it) {
        const int64_t tile = tile_begin + blockIdx.x + it * (int64_t)gridDim.x;
        const int64_t base = tile * K1_TILE;
        const int s = (int)(it % K1_STAGES);
        // the sample in front of the tile comes straight from global memory (warp 0 alone needs it; the load is
        // in flight while the warp waits for the tile)
        V before = (V)0;
        if (warp == 0 && base > 0) before = K1Key<T>::of(__ldg(x + base - 1), kxor);
        k1_mbar_wait(&S.full[s], (unsigned)((it / K1_STAGES) & 1));
        // ---- this warp's span: 4 rows of 128 samples, lane l holds samples 4l .. 4l+3 of each row ----
        T *sp = &S.stage[s][0] + warp * K1_SPAN;
        const bool ragged = base + K1_TILE > n;
        V ahead = (V)0;                                     // ragged tile: the sample in front of this warp's span
        if (ragged) {
            // last tile of the trace: nothing was staged; every warp brings its own span in (past n the last sample
            // repeats, which adds no crossing and no new extreme) and reads back only what it wrote itself
            const int64_t g0 = base + warp * K1_SPAN;
            const T fill = __ldg(x + (n - 1));
            for (int k = lane; k < K1_SPAN; k += 32) sp[k] = g0 + k < n ? __ldg(x + g0 + k) : fill;
            if (warp > 0) ahead = K1Key<T>::of(g0 - 1 < n ? __ldg(x + g0 - 1) : fill, kxor);
            __syncwarp();
        }
        V v[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if constexpr (sizeof(T) == 4) {
                const float4 q = *reinterpret_cast<const float4 *>(sp + r * 128 + lane * 4);
                v[r][0] = (T)q.x; v[r][1] = (T)q.y; v[r][2] = (T)q.z; v[r][3] = (T)q.w;
            } else if constexpr (sizeof(T) == 8) {
                const double2 q0 = *reinterpret_cast<const double2 *>(sp + r * 128 + lane * 4);
                const double2 q1 = *reinterpret_cast<const double2 *>(sp + r * 128 + lane * 4 + 2);
                v[r][0] = (T)q0.x; v[r][1] = (T)q0.y; v[r][2] = (T)q1.x; v[r][3] = (T)q1.y;
            } else {
                const uint2 q = *reinterpret_cast<const uint2 *>(sp + r * 128 + lane * 4);
                v[r][0] = K1Key<T>::of((T)(q.x & 0xffffu), kxor); v[r][1] = K1Key<T>::of((T)(q.x >> 16), kxor);
                v[r][2] = K1Key<T>::of((T)(q.y & 0xffffu), kxor); v[r][3] = K1Key<T>::of((T)(q.y >> 16), kxor);
            }
        }
        // side of the sample in front of the span
        const bool carry_below = (warp == 0 ? before : (ragged ? ahead : K1Key<T>::of(sp[-1], kxor))) < thr;
        __syncwarp();
        if (lane == 0) k1_mbar_arrive(&S.empty[s]);   // this warp has its samples in registers

        V m = v[0][0], M = v[0][0];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                m = k1_min<V>(m, v[r][k]);
                M = k1_max_nan(M, v[r][k]);
            }
        const bool w_below = __any_sync(PP_FULL, m < thr), w_above = __any_sync(PP_FULL, !(M < thr));
        const bool w_nan = __any_sync(PP_FULL, M != M);
        const int64_t r_idx = tile * K1_WARPS + warp;
        const bool first_below = __shfl_sync(PP_FULL, (int)(v[0][0] < thr), 0) != 0;
        // the very first sample of the trace never starts a new run
        const bool carry = (base == 0 && warp == 0) ? first_below : carry_below;
        if (!(w_below && w_above) && carry == w_below) {
            // ---- no crossing: the whole span continues the open run ----
            unsigned long long kmin = k1_warp_min_key(m);
            unsigned long long kmax = k1_warp_max_key(M);
            if (w_nan) { kmin = 0ull; kmax = ~0ull; }
            if (lane == 0) {
                K1Record R;
                R.count = 0u; R.first_below = first_below ? 1u : 0u; R.head_min = kmin; R.head_max = kmax;
                rec[r_idx] = R;
            }
            continue;
        }
        // ---- crossings: words of 32 below-bits (lanes 8g .. 8g+7 hold word g of a row), crossing bits, counts ----
        unsigned long long *smin = S.smin[warp], *smax = S.smax[warp];
        unsigned e[4], off[4];
        unsigned running = 0u;
        unsigned prev_top = carry ? 1u : 0u;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const unsigned nib = (v[r][0] < thr ? 1u : 0u) | (v[r][1] < thr ? 2u : 0u) | (v[r][2] < thr ? 4u : 0u) |
                                 (v[r][3] < thr ? 8u : 0u);
            unsigned w = nib << ((lane & 7) * 4);
            w |= __shfl_xor_sync(PP_FULL, w, 1);
            w |= __shfl_xor_sync(PP_FULL, w, 2);
            w |= __shfl_xor_sync(PP_FULL, w, 4);
            // top bit of the previous word: previous lane group, or the previous row's last word / the carry
            const unsigned left = __shfl_sync(PP_FULL, w, (lane & 24) - 8 < 0 ? 0 : (lane & 24) - 8) >> 31;
            const unsigned cin = (lane >> 3) == 0 ? prev_top : left;
            e[r] = w ^ ((w << 1) | cin);
            prev_top = __shfl_sync(PP_FULL, w, 31) >> 31;
            const unsigned c = __popc(e[r]);
            const unsigned c0 = __shfl_sync(PP_FULL, c, 0), c1 = __shfl_sync(PP_FULL, c, 8);
            const unsigned c2 = __shfl_sync(PP_FULL, c, 16), c3 = __shfl_sync(PP_FULL, c, 24);
            const int g = lane >> 3;
            off[r] = running + (g > 0 ? c0 : 0u) + (g > 1 ? c1 : 0u) + (g > 2 ? c2 : 0u);
            running += c0 + c1 + c2 + c3;
        }
        const unsigned count = running;
        // ---- min / max per piece: local run id of every sample = crossings up to and including its own bit.
        //      One warp reduction per piece (a handful per span) -- 64-bit shared-memory atomics per sample would
        //      serialise 512 compare-and-swap loops on two addresses (measured: the whole kernel at 2.0 TB/s) ----
        unsigned rid[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int b0 = (lane & 7) * 4;
            unsigned q = off[r] + __popc(e[r] & ((2u << b0) - 1u));
            const unsigned inner = (e[r] >> (b0 + 1)) & 7u;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k > 0) q += (inner >> (k - 1)) & 1u;
                rid[r][k] = q;
            }
        }
        const unsigned q_last = count < (unsigned)K1_STAGE ? count : (unsigned)K1_STAGE;
        for (unsigned q = 0; q <= q_last; ++q) {
            V pm = v[0][0], pM = v[0][0];
            bool have = false, pnan = false;
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool mine = rid[r][k] == q;
                    const V val = v[r][k];
                    pm = mine ? (have ? k1_min<V>(pm, val) : val) : pm;
                    pM = mine ? (have ? k1_max<V>(pM, val) : val) : pM;
                    pnan |= mine && (val != val);
                    have |= mine;
                }
            unsigned long long kmin = k1_warp_min_u64(have ? pp_dkey((double)pm) : PP_MINKEY64_EMPTY);
            unsigned long long kmax = k1_warp_max_u64(have ? pp_dkey((double)pM) : PP_MAXKEY64_EMPTY);
            if (__any_sync(PP_FULL, pnan)) { kmin = 0ull; kmax = ~0ull; }
            if (lane == 0) { smin[q] = kmin; smax[q] = kmax; }
        }
        __syncwarp();
        // ---- positions of the first K1_STAGE crossings ----
        if ((lane & 7) == 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                unsigned bits = e[r], k = off[r];
                while (bits && k < (unsigned)K1_STAGE) {
                    const int bit = __ffs(bits) - 1;
                    bits &= bits - 1;
                    staged[r_idx * K1_STAGE + k].pos = (unsigned)(r * 128 + (lane >> 3) * 32 + bit);
                    ++k;
                }
            }
        }
        __syncwarp();
        if (lane < K1_STAGE && (unsigned)lane < count) {
            staged[r_idx * K1_STAGE + lane].mn = smin[lane + 1];
            staged[r_idx * K1_STAGE + lane].mx = smax[lane + 1];
        }
        if (lane == 0) {
            K1Record R;
            R.count = count; R.first_below = first_below ? 1u : 0u; R.head_min = smin[0]; R.head_max = smax[0];
            rec[r_idx] = R;
        }
        __syncwarp();
    }
}

// One thread per span record of [rec_begin, rec_end): first run index of every span by an exclusive scan of the
// crossing counts (block scan + decoupled look-back over the blocks of THIS launch, seeded with the crossings
// found by earlier launches: ctr->n_edges), then the run starts and the min / max pieces go into the run table.
// `blk_state` holds one word per block of the launch, zeroed beforehand.
constexpr int K1B_THREADS = 256;
#define PP_TS_AGG (1ull << 62)
#define PP_TS_INC (2ull << 62)
#define PP_TS_MASK (3ull << 62)

template <typename T>
__global__ void __launch_bounds__(K1B_THREADS)
k1_stitch(const T *__restrict__ x, int64_t n, typename K1Key<T>::V thr, int kxor, int64_t rec_begin, int64_t rec_end,
          const K1Record *__restrict__ rec, const K1Staged *__restrict__ staged,
          unsigned long long *__restrict__ blk_state, PPCounters *ctr, int flip, int64_t *__restrict__ run_start,
          unsigned long long *__restrict__ run_minkey, unsigned long long *__restrict__ run_maxkey, int64_t cap_runs)
{
    __shared__ unsigned long long wtot[K1B_THREADS / 32];
    __shared__ unsigned long long s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t r = rec_begin + (int64_t)blockIdx.x * K1B_THREADS + tid;
    const bool live = r < rec_end;
    K1Record R;
    R.count = 0u; R.first_below = 0u; R.head_min = PP_MINKEY64_EMPTY; R.head_max = PP_MAXKEY64_EMPTY;
    if (live) R = rec[r];
    // crossings of the launches before this one (0 for a fresh scan).  Read from one slot, written to the other
    // (`flip` alternates per launch), so that a block starting late cannot pick up this launch's own total.
    const unsigned long long seed = ctr->n_edges[flip & 1];
    unsigned long long inc = R.count;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(PP_FULL, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    unsigned long long add = 0, total = 0;
    for (int w = 0; w < K1B_THREADS / 32; ++w) {
        if (w < warp) add += wtot[w];
        total += wtot[w];
    }
    if (warp == 0) {
        // decoupled look-back over the blocks of this launch
        unsigned long long prefix = 0;
        if (blockIdx.x == 0) {
            if (lane == 0) atomicExch(&blk_state[0], PP_TS_INC | total);
        } else {
            if (lane == 0) atomicExch(&blk_state[blockIdx.x], PP_TS_AGG | total);
            long long j = (long long)blockIdx.x - 1;
            for (;;) {
                const long long idx = j - lane;
                unsigned long long st = idx >= 0 ? pp_ld_volatile_u64(blk_state + idx) : PP_TS_INC;
                while (__any_sync(PP_FULL, (st & PP_TS_MASK) == 0ull))
                    st = idx >= 0 ? pp_ld_volatile_u64(blk_state + idx) : PP_TS_INC;
                const unsigned inc_mask = __ballot_sync(PP_FULL, (st & PP_TS_MASK) == PP_TS_INC);
                unsigned long long val = st & ~PP_TS_MASK;
                if (inc_mask) {
                    const int first = __ffs(inc_mask) - 1;
                    if (lane > first) val = 0;
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) val += __shfl_xor_sync(PP_FULL, val, d);
                prefix += val;
                if (inc_mask) break;
                j -= 32;
            }
            if (lane == 0) atomicExch(&blk_state[blockIdx.x], PP_TS_INC | (prefix + total));
        }
        if (lane == 0) s_base = seed + prefix;
    }
    __syncthreads();
    if (!live) return;
    const unsigned long long first_run = s_base + add + inc - R.count;   // the run this span's first samples belong to
    if (r == 0) {
        ctr->first_below = R.first_below;
        if (cap_runs > 0) run_start[0] = 0;
    }
    if (r == rec_end - 1) {
        ctr->n_edges[(flip & 1) ^ 1] = first_run + R.count;   // the next launch (a later chunk) continues from here
        if (rec_end * K1_SPAN >= n) ctr->n_runs = first_run + R.count + 1;   // the trace's last span
    }
    const int64_t span0 = r * K1_SPAN;
    if (R.count <= (unsigned)K1_STAGE) {
        if ((int64_t)first_run < cap_runs && R.head_min != PP_MINKEY64_EMPTY) {
            atomicMin(&run_minkey[first_run], R.head_min);
            atomicMax(&run_maxkey[first_run], R.head_max);
        }
        for (unsigned k = 0; k < R.count; ++k) {
            const K1Staged c = staged[r * K1_STAGE + k];
            const unsigned long long rid = first_run + k + 1;
            if ((int64_t)rid < cap_runs) {
                run_start[rid] = span0 + c.pos;
                atomicMin(&run_minkey[rid], c.mn);
                atomicMax(&run_maxkey[rid], c.mx);
            }
        }
        return;
    }
    // ---- more crossings than were staged (noise riding on the threshold): walk the span again ----
    unsigned long long rid = first_run;
    bool below = K1Key<T>::of(__ldg(x + (span0 > 0 ? span0 - 1 : 0)), kxor) < thr;
    unsigned long long kmin = PP_MINKEY64_EMPTY, kmax = PP_MAXKEY64_EMPTY;
    const int64_t end = span0 + K1_SPAN < n ? span0 + K1_SPAN : n;
    for (int64_t p = span0; p < end; ++p) {
        const typename K1Key<T>::V val = K1Key<T>::of(__ldg(x + p), kxor);
        const bool b = val < thr;
        if (b != below) {
            if ((int64_t)rid < cap_runs && kmin != PP_MINKEY64_EMPTY) {
                atomicMin(&run_minkey[rid], kmin);
                atomicMax(&run_maxkey[rid], kmax);
            }
            ++rid;
            if ((int64_t)rid < cap_runs) run_start[rid] = p;
            kmin = PP_MINKEY64_EMPTY; kmax = PP_MAXKEY64_EMPTY;
            below = b;
        }
        const bool isn = val != val;
        const unsigned long long k = pp_dkey((double)val);
        const unsigned long long lo = isn ? 0ull : k, hi = isn ? ~0ull : k;
        kmin = lo < kmin ? lo : kmin;
        kmax = hi > kmax ? hi : kmax;
    }
    if ((int64_t)rid < cap_runs && kmin != PP_MINKEY64_EMPTY) {
        atomicMin(&run_minkey[rid], kmin);
        atomicMax(&run_maxkey[rid], kmax);
    }
}

__device__ __forceinline__ double pp_decode_min64(unsigned long long k)
{
    if (k == 0ull || k == PP_MINKEY64_EMPTY) return __longlong_as_double(0x7ff8000000000000LL);
    return pp_dkey_inv(k);
}
__device__ __forceinline__ double pp_decode_max64(unsigned long long k)
{
    if (k == ~0ull || k == PP_MAXKEY64_EMPTY) return __longlong_as_double(0x7ff8000000000000LL);
    return pp_dkey_inv(k);
}

// Decode the run table: length, side, min/max as float64 (what the rules see).  adc != 0: the keys are ADC keys
// c ^ kxor, decoded with `a` (the current is non-decreasing in the key, so the extreme keys give the extremes).
__global__ void __launch_bounds__(256)
k1_finalize_runs(int64_t n, const PPCounters *ctr, const int64_t *__restrict__ run_start,
                 const unsigned long long *__restrict__ run_minkey,
                 const unsigned long long *__restrict__ run_maxkey,
                 int64_t cap_runs, int64_t *__restrict__ run_len, double *__restrict__ run_min,
                 double *__restrict__ run_max, unsigned char *__restrict__ run_below, int adc, PPAdc a)
{
    const int kxor = a.scale < 0.0 ? -1 : 0;
    int64_t n_runs = (int64_t)ctr->n_runs;
    if (n_runs > cap_runs) n_runs = cap_runs;
    const unsigned first_below = ctr->first_below;
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_runs;
         r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = run_start[r];
        const int64_t e = (r + 1 < (int64_t)ctr->n_runs && r + 1 < cap_runs) ? run_start[r + 1] : n;
        run_len[r] = e - s;
        double mn = pp_decode_min64(run_minkey[r]), mx = pp_decode_max64(run_maxkey[r]);
        if (adc) {   // (an empty run stays NaN)
            if (mn == mn) mn = pp_adc_decode((int)mn ^ kxor, a);
            if (mx == mx) mx = pp_adc_decode((int)mx ^ kxor, a);
        }
        run_min[r] = mn;
        run_max[r] = mx;
        run_below[r] = (unsigned char)((first_below ^ (unsigned)(r & 1)) & 1u);
    }
}

// _lambda_select for the default-shaped rules + compaction into the event
// table (ev_start, ev_len, ev_off = exclusive prefix of lengths).  One CTA;
// the run table is tiny next to the trace.
constexpr int SEL_THREADS = 1024;

__global__ void __launch_bounds__(SEL_THREADS)
k1_select_events(PPCounters *ctr, const int64_t *__restrict__ run_start,
                 const int64_t *__restrict__ run_len, const double *__restrict__ run_min,
                 const double *__restrict__ run_max, int64_t cap_runs, int rule_mask,
                 int64_t duration_gt, int64_t duration_lt, double min_gt, double max_lt,
                 int skip_first, int skip_last, int64_t *__restrict__ ev_start,
                 int64_t *__restrict__ ev_len, int64_t *__restrict__ ev_off, int64_t cap_events,
                 int incremental /* 0: whole run table; 1: append the runs completed since the last call,
                                    the still open last run excluded; 2: same, last call (open run included) */,
                 const long long *__restrict__ plan = nullptr /* multi-GPU: k_shard_plan's record overrides
                                                                 skip_first / skip_last */)
{
    if (plan) { skip_first = (int)plan[0]; skip_last = (int)plan[1]; }
    __shared__ unsigned wcnt[SEL_THREADS / 32];
    __shared__ long long wlen[SEL_THREADS / 32];
    __shared__ unsigned long long s_cnt_carry;
    __shared__ long long s_len_carry;
    __shared__ unsigned s_cnt_total;
    __shared__ long long s_len_total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t n_runs = (int64_t)ctr->n_runs;
    if (n_runs > cap_runs) n_runs = cap_runs;
    int64_t r_begin = 0;
    const unsigned long long ev_before = incremental ? ctr->n_events : 0ull;
    if (incremental) {
        r_begin = (int64_t)ctr->sel_next_run;
        if (incremental == 1 && n_runs > 0) n_runs -= 1;
        if (n_runs < r_begin) n_runs = r_begin;
    }
    if (tid == 0) {
        s_cnt_carry = ev_before;
        s_len_carry = incremental ? (long long)ctr->n_event_samples : 0;
    }
    __syncthreads();
    // one run per thread and trip, coalesced; the next trip's rows are requested before this trip's scan, so that a
    // trip costs its two barriers and not a round trip to memory (a single SM serves this kernel: eight strided rows
    // per thread had its load unit queue 25 k line requests, 25 us for 10^4 runs)
    auto fetch = [&](int64_t r, long long &len, double &mn, double &mx, long long &st) {
        const bool in = r < n_runs;
        len = in ? run_len[r] : 0;
        st = in ? run_start[r] : 0;
        mn = in && (rule_mask & PP_RULE_MIN_GT) ? run_min[r] : 0.0;
        mx = in && (rule_mask & PP_RULE_MAX_LT) ? run_max[r] : 0.0;
    };
    long long len_n, st_n;
    double mn_n, mx_n;
    fetch(r_begin + tid, len_n, mn_n, mx_n, st_n);
    for (int64_t c0 = r_begin; c0 < n_runs; c0 += SEL_THREADS) {
        const int64_t r = c0 + tid;
        const long long len = len_n, st = st_n;
        const double mn = mn_n, mx = mx_n;
        fetch(r + SEL_THREADS, len_n, mn_n, mx_n, st_n);
        bool keep = r < n_runs;
        if (rule_mask & PP_RULE_DURATION_GT) keep = keep && (len > duration_gt);
        if (rule_mask & PP_RULE_DURATION_LT) keep = keep && (len < duration_lt);
        if (rule_mask & PP_RULE_MIN_GT) keep = keep && (mn > min_gt);
        if (rule_mask & PP_RULE_MAX_LT) keep = keep && (mx < max_lt);
        if (skip_first && r == 0) keep = false;
        if (skip_last && r == n_runs - 1) keep = false;
        unsigned c = keep ? 1u : 0u;
        long long l = keep ? len : 0;
        unsigned ci = c;
        long long li = l;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned tc = __shfl_up_sync(PP_FULL, ci, d);
            long long tl = __shfl_up_sync(PP_FULL, li, d);
            if (lane >= d) { ci += tc; li += tl; }
        }
        if (lane == 31) { wcnt[warp] = ci; wlen[warp] = li; }
        __syncthreads();
        if (warp == 0) {   // exclusive scan of the 32 warp totals by one warp (a loop per thread cost 100 instructions a trip)
            unsigned wc = wcnt[lane], wci = wc;
            long long wl = wlen[lane], wli = wl;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                unsigned tc = __shfl_up_sync(PP_FULL, wci, d);
                long long tl = __shfl_up_sync(PP_FULL, wli, d);
                if (lane >= d) { wci += tc; wli += tl; }
            }
            wcnt[lane] = wci - wc;
            wlen[lane] = wli - wl;
            if (lane == 31) { s_cnt_total = wci; s_len_total = wli; }
        }
        __syncthreads();
        const unsigned long long idx = s_cnt_carry + wcnt[warp] + (ci - c);
        const long long off = s_len_carry + wlen[warp] + (li - l);
        if (keep && (int64_t)idx < cap_events) {
            ev_start[idx] = st;
            ev_len[idx] = len;
            ev_off[idx] = off;
        }
        __syncthreads();
        if (tid == 0) {
            s_cnt_carry += s_cnt_total;
            s_len_carry += s_len_total;
        }
        __syncthreads();
    }
    if (tid == 0) {
        unsigned long long ne = s_cnt_carry;
        if ((int64_t)ne > cap_events) { ne = cap_events; atomicOr(&ctr->overflow, PP_OVF_RUNS); }
        ctr->n_events = ne;
        ctr->n_event_samples = (unsigned long long)s_len_carry;
        ctr->sel_next_run = (unsigned long long)n_runs;
        ctr->ev_begin = ev_before < ne ? ev_before : ne;
        ev_off[ne] = s_len_carry;
    }
}

// Host-chosen events: exclusive prefix of the lengths (same single-CTA scan).
__global__ void __launch_bounds__(SEL_THREADS)
k1_event_offsets(PPCounters *ctr, const int64_t *__restrict__ ev_len, int64_t n_events,
                 int64_t *__restrict__ ev_off)
{
    __shared__ long long wlen[SEL_THREADS / 32];
    __shared__ long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int64_t c0 = 0; c0 < n_events; c0 += SEL_THREADS) {
        const int64_t r = c0 + tid;
        long long l = r < n_events ? ev_len[r] : 0;
        long long li = l;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            long long tl = __shfl_up_sync(PP_FULL, li, d);
            if (lane >= d) li += tl;
        }
        if (lane == 31) wlen[warp] = li;
        __syncthreads();
        long long lb = 0;
        for (int w = 0; w < warp; ++w) lb += wlen[w];
        const long long off = s_carry + lb + (li - l);
        if (r < n_events) ev_off[r] = off;
        __syncthreads();
        if (tid == SEL_THREADS - 1) s_carry = off + l;
        __syncthreads();
    }
    if (tid == 0) {
        ev_off[n_events] = s_carry;
        ctr->n_events = (unsigned long long)n_events;
        ctr->n_event_samples = (unsigned long long)s_carry;
        ctr->ev_begin = 0;
        ctr->overflow &= ~(unsigned)PP_OVF_FILTER_SHORT;  // a refused filter spoke of the previous events
    }
}

// Multi-GPU: the record a rank publishes about its chunk (pypore_b200/dist.py boundary_info):
// [n_local, n_runs, first_below, first_len, first_min, first_max,
//  last_below, last_start, last_len, last_min, last_max, run-table-overflow flag]
__global__ void k1_boundary_record(int64_t n_local, const PPCounters *ctr, const int64_t *__restrict__ run_start,
                                   const int64_t *__restrict__ run_len, const double *__restrict__ run_min,
                                   const double *__restrict__ run_max, const unsigned char *__restrict__ run_below,
                                   int64_t cap_runs, double *__restrict__ rec)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int64_t n_runs = (int64_t)ctr->n_runs;
    const bool ovf = n_runs > cap_runs || n_runs <= 0;
    const int64_t last = ovf ? 0 : n_runs - 1;
    rec[0] = (double)n_local;
    rec[1] = (double)n_runs;
    rec[2] = (double)run_below[0];
    rec[3] = (double)run_len[0];
    rec[4] = run_min[0];
    rec[5] = run_max[0];
    rec[6] = (double)run_below[last];
    rec[7] = (double)run_start[last];
    rec[8] = (double)run_len[last];
    rec[9] = run_min[last];
    rec[10] = run_max[last];
    rec[11] = ovf ? 1.0 : 0.0;
}

// Multi-GPU: this rank's row of dist.py plan_boundaries, derived on the DEVICE from the all-gathered
// boundary records (infos[q] = rank q's k1_boundary_record), so that a step needs no host round trip
// between the threshold scan and the split search.  `halo_avail` continuation samples of the right
// neighbour were placed after the chunk speculatively, before anything was known about the runs.
// plan = [skip_first, skip_last, has_event, ev_start, ev_len, redo, halo samples needed, 0]:
//   redo = PP_OVF_HALO when the straddling event this rank owns needs more than halo_avail samples
//          (or continues past the right neighbour), PP_OVF_RUNS when any rank's run table overflowed;
//          the host then repeats the step with the host-planned exchange (dist.py).
constexpr int PP_PLAN_WORDS = 8;

__device__ __forceinline__ double pp_nan_min(double a, double b) { return (a != a || b != b) ? a + b : (a < b ? a : b); }
__device__ __forceinline__ double pp_nan_max(double a, double b) { return (a != a || b != b) ? a + b : (a > b ? a : b); }

__global__ void k_shard_plan(const double *__restrict__ infos, int rank, int world, int rule_mask,
                             int64_t duration_gt, int64_t duration_lt, double min_gt, double max_lt,
                             int64_t halo_avail, long long *__restrict__ plan)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int L = 12;
    auto joins = [&](int q) { return infos[q * L + 6] == infos[(q + 1) * L + 2]; };  // last_below == next first_below
    long long redo = 0;
    for (int q = 0; q < world; ++q)
        if (infos[q * L + 11] != 0.0) redo |= PP_OVF_RUNS;
    const bool skip_first = rank > 0 && joins(rank - 1);
    bool skip_last = false;
    long long has_event = 0, ev_start = 0, ev_len = 0, need = 0;
    if (rank < world - 1 && joins(rank)) {
        skip_last = true;
        const double *me = infos + rank * L;
        const bool owns = !(me[1] == 1.0 && skip_first);  // else the run started further left
        if (owns) {
            long long length = (long long)me[8];
            double mn = me[9], mx = me[10];
            int q = rank + 1;
            for (;;) {
                const double *o = infos + q * L;
                length += (long long)o[3];
                mn = pp_nan_min(mn, o[4]);
                mx = pp_nan_max(mx, o[5]);
                if (o[1] == 1.0 && q < world - 1 && joins(q)) { ++q; continue; }
                break;
            }
            bool ok = true;
            if (rule_mask & PP_RULE_DURATION_GT) ok = ok && (length > duration_gt);
            if (rule_mask & PP_RULE_DURATION_LT) ok = ok && (length < duration_lt);
            if (rule_mask & PP_RULE_MIN_GT) ok = ok && (mn > min_gt);
            if (rule_mask & PP_RULE_MAX_LT) ok = ok && (mx < max_lt);
            if (ok) {
                need = length - (long long)me[8];
                if (q == rank + 1 && need <= halo_avail) {
                    has_event = 1;
                    ev_start = (long long)me[7];
                    ev_len = length;
                } else {
                    redo |= PP_OVF_HALO;
                }
            }
        }
    }
    plan[0] = skip_first;
    plan[1] = skip_last;
    plan[2] = has_event;
    plan[3] = ev_start;
    plan[4] = ev_len;
    plan[5] = redo;
    plan[6] = need;
    plan[7] = 0;
}

// The straddling event of k_shard_plan appended after the selected events.
__global__ void k_append_planned_event(PPCounters *ctr, int64_t *ev_start, int64_t *ev_len, int64_t *ev_off,
                                       int64_t cap_events, const long long *__restrict__ plan)
{
    if (blockIdx.x != 0 || threadIdx.x != 0 || !plan[2]) return;
    const unsigned long long e = ctr->n_events;
    if ((int64_t)e >= cap_events) { atomicOr(&ctr->overflow, PP_OVF_RUNS); return; }
    ev_start[e] = plan[3];
    ev_len[e] = plan[4];
    ev_off[e + 1] = ev_off[e] + plan[4];  // ev_off[e] already holds the running total
    ctr->n_events = e + 1;
    ctr->n_event_samples += (unsigned long long)plan[4];
}

// Multi-GPU: [n_runs, n_events, n_event_samples, n_segments, overflow flags, candidates, scans, exact]
__global__ void k_result_record(const PPCounters *ctr, long long *__restrict__ rec,
                                const long long *__restrict__ plan = nullptr)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    rec[0] = (long long)ctr->n_runs;
    rec[1] = (long long)ctr->n_events;
    rec[2] = (long long)ctr->n_event_samples;
    rec[3] = (long long)ctr->n_segments;
    rec[4] = (long long)ctr->overflow | (plan ? plan[5] : 0);
    rec[5] = (long long)ctr->n_cand;
    rec[6] = (long long)ctr->n_scan;
    rec[7] = (long long)ctr->n_exact;
}

// Multi-GPU: event and segment tables packed into 8-byte words for ONE all-gather:
// n_events rows {global start, length}, then n_segments rows of PP_SEG_WORDS words
//   { global event id (low 32 bits) | event-relative start (high 32 bits),  mean,  std,  min | max as float32 }
// -- 32 B instead of the table's 56: `end` is the next row's start (or the event's length) and is rebuilt
// after the gather, the sharded path works on float32 traces so min / max are float32 values, and an event
// is shorter than 2^31 samples.  Counts and the global event-id base come from the all-gathered result
// records in DEVICE memory (rec_all[r] = rank r's k_result_record), so the host does not have to know them yet.
constexpr int PP_SEG_WORDS = 4;

__global__ void __launch_bounds__(256)
k_pack_tables(const long long *__restrict__ rec_all, int rank, int64_t cap_words, int64_t sample_offset,
              const int64_t *__restrict__ ev_start, const int64_t *__restrict__ ev_len,
              const int *__restrict__ seg_event, const int64_t *__restrict__ seg_start,
              const int64_t *__restrict__ seg_end, const double *__restrict__ mean,
              const double *__restrict__ sd, const double *__restrict__ mn, const double *__restrict__ mx,
              long long *__restrict__ out)
{
    const int64_t n_events = rec_all[8 * rank + 1], n_segments = rec_all[8 * rank + 3];
    if (2 * n_events + PP_SEG_WORDS * n_segments > cap_words) return;  // the host notices from the same records and retries
    int64_t event_base = 0;
    for (int r = 0; r < rank; ++r) event_base += rec_all[8 * r + 1];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t e = t0; e < n_events; e += stride) {
        out[2 * e] = ev_start[e] + sample_offset;
        out[2 * e + 1] = ev_len[e];
    }
    longlong2 *seg = reinterpret_cast<longlong2 *>(out + 2 * n_events);  // 16-byte aligned: 2 words per event
    for (int64_t k = t0; k < n_segments; k += stride) {
        const unsigned long long id = (unsigned long long)((long long)seg_event[k] + event_base) & 0xffffffffull;
        const unsigned long long st = (unsigned long long)seg_start[k] << 32;
        const unsigned long long lo = (unsigned long long)__float_as_uint((float)mn[k]);
        const unsigned long long hi = (unsigned long long)__float_as_uint((float)mx[k]) << 32;
        seg[2 * k] = make_longlong2((long long)(id | st), __double_as_longlong(mean[k]));
        seg[2 * k + 1] = make_longlong2(__double_as_longlong(sd[k]), (long long)(lo | hi));
    }
}

// Multi-GPU: the all-gathered packed tables (row r of `g`, `m` words long, = rank r's k_pack_tables output) unpacked
// into the caller's tables in ONE pass, one contiguous array per column -- events {global start, length}, segments
// {global event id, start, end, mean, std, min, max} -- written straight into page-locked host memory
// (device-visible aliases) or into device memory; consecutive threads write consecutive 8-byte elements, so every
// store is a full line on its way over PCIe (rows of 24 + 32 bytes written per thread ran at 7 GB/s).  `end` is
// the next row's start inside the same event, else the event's length.  Counts come from the all-gathered result
// records on the device (rec_all[8 r + 1] events, rec_all[8 r + 3] segments of rank r).  The first version did
// this with a dozen eager torch operations over 2.4 M rows followed by pageable copies: 60 of the 77 ms of an
// 8-GPU end-to-end step.
constexpr int PP_MAX_WORLD = 64;

struct PPUnpacked {
    int64_t cap_events, cap_segments;
    long long *ev_start, *ev_len;
    long long *seg_event, *seg_start, *seg_end;
    double *mean, *sd, *mn, *mx;
};

__global__ void __launch_bounds__(256)
k_unpack_tables(const long long *__restrict__ g, int world, int64_t m, const long long *__restrict__ rec_all,
                int rank_lo, int rank_hi, PPUnpacked O, unsigned *__restrict__ status)
{
    __shared__ long long e_base[PP_MAX_WORLD + 1], s_base[PP_MAX_WORLD + 1];
    if (threadIdx.x == 0) {
        long long e = 0, sg = 0;
        for (int r = 0; r < world; ++r) {
            e_base[r] = e; s_base[r] = sg;
            e += rec_all[8 * r + 1];
            sg += rec_all[8 * r + 3];
        }
        e_base[world] = e; s_base[world] = sg;
    }
    __syncthreads();
    // rows of the ranks [rank_lo, rank_hi) only, written from index 0 (event ids and starts stay global)
    const long long E0 = e_base[rank_lo], S0 = s_base[rank_lo];
    const long long E = e_base[rank_hi], S = s_base[rank_hi];
    if (E - E0 > O.cap_events || S - S0 > O.cap_segments) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(status, 1u);
        return;
    }
    O.ev_start -= E0; O.ev_len -= E0;
    O.seg_event -= S0; O.seg_start -= S0; O.seg_end -= S0;
    O.mean -= S0; O.sd -= S0; O.mn -= S0; O.mx -= S0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t k = E0 + t0; k < E; k += stride) {
        int r = rank_lo;
        while (k >= e_base[r + 1]) ++r;
        const long long *row = g + (int64_t)r * m + 2 * (k - e_base[r]);
        O.ev_start[k] = row[0];
        O.ev_len[k] = row[1];
    }
    for (int64_t k = S0 + t0; k < S; k += stride) {
        int r = rank_lo;
        while (k >= s_base[r + 1]) ++r;
        const long long n_ev = e_base[r + 1] - e_base[r], n_sg = s_base[r + 1] - s_base[r];
        const long long j = k - s_base[r];
        const long long *gr = g + (int64_t)r * m;
        const longlong2 *seg = reinterpret_cast<const longlong2 *>(gr + 2 * n_ev);
        const longlong2 a = seg[2 * j], b = seg[2 * j + 1];
        const long long event = a.x & 0xffffffffLL, start = (long long)((unsigned long long)a.x >> 32);
        long long end;
        bool same = false;
        long long nxt = 0;
        if (j + 1 < n_sg) {
            nxt = seg[2 * (j + 1)].x;
            same = (nxt & 0xffffffffLL) == event;
        }
        if (same) end = (long long)((unsigned long long)nxt >> 32);
        else end = gr[2 * (event - e_base[r]) + 1];   // the event's length (events of rank r carry ids e_base[r] ..)
        O.seg_event[k] = event;
        O.seg_start[k] = start;
        O.seg_end[k] = end;
        O.mean[k] = __longlong_as_double(a.y);
        O.sd[k] = __longlong_as_double(b.x);
        O.mn[k] = (double)__uint_as_float((unsigned)((unsigned long long)b.y & 0xffffffffull));
        O.mx[k] = (double)__uint_as_float((unsigned)((unsigned long long)b.y >> 32));
    }
}

// Multi-GPU control exchange without a collective: the few dozen bytes every rank must know about every other rank
// (boundary records after the scan, result records after the search) travel as plain stores over NVLink into a
// small buffer on EVERY peer (mapped through CUDA IPC), followed by a flag; the same kernel then waits for the
// flags of all ranks in its own buffer and copies the records out.  One 64-thread launch on the step's stream
// instead of an NCCL all-gather (whose launch latency, not its bandwidth, sat on the critical path: 0.04 ms per
// all-gather at 8 GPUs, two per step).
//   buffer layout: [parity 0 | parity 1] x [world slots] x PP_CTL_SLOT words; slot = 16 payload words, word 31 = flag.
//   `seq` increases by one per exchange on every rank alike; exchange seq uses the slots of parity seq & 1.  A rank
//   can only reach exchange seq + 2 after every rank has published seq + 1, i.e. after every rank has finished
//   reading seq (stream order on each rank), so two parities suffice.
constexpr int PP_CTL_SLOT = 32;
constexpr int PP_CTL_PAYLOAD = 16;
constexpr long long PP_CTL_SPINS = 4000000;   // ~ seconds: a dead peer must not hang the device

__global__ void __launch_bounds__(64)
k_ctl_exchange(unsigned long long *const *__restrict__ peers, int rank, int world, unsigned long long seq,
               const unsigned long long *__restrict__ src, int n_words, unsigned long long *__restrict__ dst,
               PPCounters *ctr)
{
    const int q = threadIdx.x;
    if (q >= world) return;
    const size_t par = (size_t)(seq & 1ull) * (size_t)world;
    {   // publish: my record into slot `rank` of peer q's buffer, then the flag
        volatile unsigned long long *slot = peers[q] + (par + (size_t)rank) * PP_CTL_SLOT;
        for (int k = 0; k < n_words; ++k) slot[k] = src[k];
        __threadfence_system();
        slot[PP_CTL_SLOT - 1] = seq;
    }
    {   // collect: rank q's record from slot q of my own buffer
        volatile unsigned long long *slot = peers[rank] + (par + (size_t)q) * PP_CTL_SLOT;
        long long spins = 0;
        while (slot[PP_CTL_SLOT - 1] != seq) {
            if (++spins > PP_CTL_SPINS) { atomicOr(&ctr->overflow, (unsigned)PP_OVF_CTL); break; }
            __nanosleep(200);
        }
        __threadfence_system();
        for (int k = 0; k < n_words; ++k) dst[(size_t)q * n_words + k] = slot[k];
    }
}
