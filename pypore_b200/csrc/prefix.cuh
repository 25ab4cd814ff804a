// prefix.cuh -- K2: FastStatSplit's cumsums (PyPore/cparsers.pyx:110-111).
//
//   c  = np.cumsum(x)          c2 = np.cumsum(x * x)        (fp64, restart per event)
//
// stored interleaved as double2 {c, c2} per event sample in "flat event space"
// (event e occupies [ev_off[e], ev_off[e+1])).
//
// np.cumsum is a strictly sequential fp64 accumulation and the split decisions
// downstream are compared bit-exactly, so two kernels cooperate:
//   * k2_prefix_tiled: a per-event tiled scan with decoupled look-back that ALSO
//     proves, with error-free TwoSum residuals, whether every addition it made was
//     exact.  If all of an event's additions were exact, every prefix value is the
//     exact real sum and therefore equals what the sequential order produces
//     (induction over i: c[i-1] exact and representable, c[i-1]+x[i] exact and
//     representable => fl() returns it).  ADC-quantised traces (real .abf data are
//     int16 counts, read_abf.py:208-210) always pass.
//   * k2_prefix_sequential: strict np.cumsum order, one thread per event, run for
//     the events the tiled scan flagged inexact (PP_PREFIX_AUTO) or for all
//     events (PP_PREFIX_SEQUENTIAL).
#pragma once
#include "common.cuh"

// Strict left-to-right order (np.cumsum's), one WARP per event: the lanes stage a tile of
// samples (and their squares) in shared memory with coalesced loads, lane 0 / lane 1 run the two
// dependent addition chains  c += x  and  c2 += x*x  over the tile (operands come from shared
// memory, so only the fp64 add latency is on the critical path), and all lanes write the tile
// of prefix sums back coalesced.  Used for the events the tiled scan could not prove exact
// (filtered float64 currents, raw non-ADC data) and for PP_PREFIX_SEQUENTIAL.
constexpr int K2S_WARPS = 8;
constexpr int K2S_TILE = 256;  // samples per warp tile

// one lane's samples of the tile starting at `base` (coalesced: sample k * 32 + lane), 0 past the end;
// kept in their own type so that nothing waits for the loads until the values are used
template <typename T>
__device__ __forceinline__ void k2s_load(const T *__restrict__ p, int64_t base, int64_t len, int lane,
                                         T (&xv)[K2S_TILE / 32])
{
#pragma unroll
    for (int k = 0; k < K2S_TILE / 32; ++k) {
        const int64_t j = base + k * 32 + lane;
        xv[k] = j < len ? __ldg(p + j) : (T)0;
    }
}

template <typename T>
__device__ __forceinline__ void k2s_event(const T *__restrict__ p, int64_t len, double2 *__restrict__ out,
                                          double (*v)[K2S_TILE], int lane, const PPAdc &adc)
{
    double acc = 0.0;  // lane 0: c, lane 1: c2
    T xv[K2S_TILE / 32], xn[K2S_TILE / 32];
    k2s_load(p, 0, len, lane, xv);
    for (int64_t base = 0; base < len; base += K2S_TILE) {
        const int cnt = (int)((len - base) < K2S_TILE ? (len - base) : K2S_TILE);
#pragma unroll
        for (int k = 0; k < K2S_TILE / 32; ++k) {
            const double x = pp_val(xv[k], adc);
            v[0][k * 32 + lane] = x;
            v[1][k * 32 + lane] = __dmul_rn(x, x);
        }
        // the next tile's samples travel while lanes 0/1 walk the chain
        if (base + K2S_TILE < len) k2s_load(p, base + K2S_TILE, len, lane, xn);
        __syncwarp();
        if (lane < 2) {
            double *q = v[lane];
            for (int j0 = 0; j0 < K2S_TILE; j0 += 16) {
                double t[16];  // operands first: their loads do not wait for the chain's stores
#pragma unroll
                for (int k = 0; k < 16; ++k) t[k] = q[j0 + k];
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    acc = __dadd_rn(acc, t[k]);
                    t[k] = acc;
                }
#pragma unroll
                for (int k = 0; k < 16; ++k) q[j0 + k] = t[k];
            }
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < K2S_TILE / 32; ++k) {
            const int j = k * 32 + lane;
            if (j < cnt) out[base + j] = make_double2(v[0][j], v[1][j]);
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < K2S_TILE / 32; ++k) xv[k] = xn[k];
    }
}

__global__ void __launch_bounds__(K2S_WARPS * 32, 3)
k2_prefix_sequential(PPSource src, const int64_t *__restrict__ ev_len, PPCounters *ctr,
                     const unsigned *__restrict__ inexact /* nullable: redo only flagged events */,
                     double2 *__restrict__ cc)
{
    __shared__ double sv[K2S_WARPS][2][K2S_TILE];  // [warp][0: x -> c, 1: x*x -> c2][sample]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t warps = (int64_t)gridDim.x * K2S_WARPS;
    // events are dealt to CTAs round-robin so that a few flagged events still spread over all SMs
    for (int64_t e = (int64_t)ctr->ev_begin + (int64_t)warp * gridDim.x + blockIdx.x; e < n_events; e += warps) {
        if (inexact) {
            if (inexact[e] == 0u) continue;
            if (lane == 0) atomicAdd(&ctr->n_seq_redo, 1ull);
        }
        const int64_t len = ev_len[e];
        const int64_t off = src.ev_off[e];
        if (src.kind == PP_SRC_TRACE32) k2s_event(src.trace + src.ev_start[e], len, cc + off, sv[warp], lane, src.adc);
        else if (src.kind == PP_SRC_TRACE64) k2s_event(src.trace64 + src.ev_start[e], len, cc + off, sv[warp], lane, src.adc);
        else if (src.kind == PP_SRC_ADC16) k2s_event(src.trace16 + src.ev_start[e], len, cc + off, sv[warp], lane, src.adc);
        else k2s_event(src.flat + off, len, cc + off, sv[warp], lane, src.adc);
    }
}


// ---------------------------------------------------------------------------
// Tiled scan with exactness proof (reduce-then-scan, no inter-CTA dependencies).
//
// Tiles never straddle events: event e owns tiles [ev_tile_off[e], ev_tile_off[e+1]) of
// K2_TILE samples each.  Three stream-ordered kernels:
//   k2_tile_reduce    per tile: sum of x and of x*x, and the exponent statistics below
//   k2_event_carries  per event: exclusive prefix of its tiles' sums, exactness verdict
//   k2_tile_scan      per tile: scan with the known carry, 16 B written per sample
// The samples are read twice (4 B each time, the second time mostly from L2); in exchange no
// CTA ever waits for another one.
//
// Exactness proof (order independent).  Let q = 2^elow be the coarsest power of two that
// divides every summand of an event (elow = min over samples of the position of the lowest
// set mantissa bit) and 2^(emax+1) a bound on every |summand|.  Any sum of a subset of the
// n summands is a multiple of q of magnitude < n * 2^(emax+1); if
//         ceil(log2 n) + emax + 1 - elow <= 53
// every such sum is exactly representable, so every partial sum of ANY summation order --
// this scan's and np.cumsum's sequential one -- is computed without rounding and the two
// agree bit for bit.  The test is evaluated separately for x and for fl(x*x).  For float32
// samples x*x is exact in fp64 (24 x 24 mantissa bits), its lowest set bit is exactly twice
// that of x and its magnitude exponent is at most 2 emax + 1, so only x is analysed.
// Events that fail the test (or contain inf/NaN) are redone by k2_prefix_sequential.
// ---------------------------------------------------------------------------
constexpr int K2_THREADS = 256;
constexpr int K2_ITEMS = 8;
constexpr int K2_TILE = K2_THREADS * K2_ITEMS;  // 2048 samples
constexpr int K2_PAD = K2_ITEMS + 1;

struct K2TileState {
    double agg_c, agg_c2;      // sum over this tile
    double carry_c, carry_c2;  // sum over all earlier tiles of the event
};

struct K2EventBits {  // per event: quantum / magnitude exponents of x and of x*x
    int elow1, emax1, elow2, emax2;
};

#define K2_ELOW_INIT 0x7fffffff
#define K2_EMAX_INIT (-0x7fffffff)
#define K2_BAD_EXP 100000

// lowest-set-bit exponent and magnitude exponent of a double (0.0 contributes nothing)
__device__ __forceinline__ void k2_exponents(double v, int &elow, int &emax)
{
    const long long b = __double_as_longlong(v);
    const int E = (int)((b >> 52) & 0x7ff);
    unsigned long long m = (unsigned long long)b & 0x000fffffffffffffULL;
    if (E == 0x7ff) { elow = -K2_BAD_EXP; emax = K2_BAD_EXP; return; }  // inf / NaN: never "exact"
    if (E == 0) {
        if (m == 0) { elow = K2_ELOW_INIT; emax = K2_EMAX_INIT; return; }
        elow = -1074 + (__ffsll((long long)m) - 1);
        emax = -1023;
        return;
    }
    m |= 0x0010000000000000ULL;
    elow = E - 1023 - 52 + (__ffsll((long long)m) - 1);
    emax = E - 1023;
}

// same for a float32 sample, 32-bit arithmetic only
__device__ __forceinline__ void k2_exponents(float v, int &elow, int &emax)
{
    const unsigned b = __float_as_uint(v);
    const int E = (int)((b >> 23) & 0xff);
    unsigned m = b & 0x007fffffu;
    if (E == 0xff) { elow = -K2_BAD_EXP; emax = K2_BAD_EXP; return; }
    if (E == 0) {
        if (m == 0) { elow = K2_ELOW_INIT; emax = K2_EMAX_INIT; return; }
        elow = -149 + (__ffs((int)m) - 1);
        emax = -127;
        return;
    }
    m |= 0x00800000u;
    elow = E - 127 - 23 + (__ffs((int)m) - 1);
    emax = E - 127;
}

struct K2Exp {
    int el1, em1, el2, em2;
    __device__ __forceinline__ void init() { el1 = el2 = K2_ELOW_INIT; em1 = em2 = K2_EMAX_INIT; }
    __device__ __forceinline__ void add(float x)
    {
        int a, b;
        k2_exponents(x, a, b);
        el1 = min(el1, a); em1 = max(em1, b);
    }
    __device__ __forceinline__ void add(double x)
    {
        int a, b;
        k2_exponents(x, a, b);
        el1 = min(el1, a); em1 = max(em1, b);
        k2_exponents(__dmul_rn(x, x), a, b);
        el2 = min(el2, a); em2 = max(em2, b);
    }
    __device__ __forceinline__ void warp_reduce()
    {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            el1 = min(el1, __shfl_xor_sync(PP_FULL, el1, d)); em1 = max(em1, __shfl_xor_sync(PP_FULL, em1, d));
            el2 = min(el2, __shfl_xor_sync(PP_FULL, el2, d)); em2 = max(em2, __shfl_xor_sync(PP_FULL, em2, d));
        }
    }
};

// ---------------------------------------------------------------------------
// Short events (<= K2F_MAX_LEN samples -- every event of the C1/C2/C3/C5 workloads): ONE pass, one
// WARP per event, no CTA barrier and no inter-CTA dependency.  The warp walks its event in steps of
// 256 samples: coalesced loads -> per-warp shared-memory transpose -> 8 consecutive samples per lane
// -> warp scan of the lane totals -> running carry in registers -> per-warp transpose -> coalesced
// 16 B stores.  The samples are read once (4 + 16 B per sample instead of 4 + 4 + 16), the exponent
// statistics of the exactness proof are gathered in the same pass and the verdict is written when the
// event ends.  Longer events keep the multi-CTA reduce / carries / scan kernels below (a single warp
// would serialise them); k2_tile_offsets gives short events no tiles.
// ---------------------------------------------------------------------------
constexpr int K2F_WARPS = 8;
constexpr int K2F_ITEMS = 8;                      // consecutive samples per lane
constexpr int K2F_TILE = 32 * K2F_ITEMS;           // samples per warp step
constexpr int K2F_PAD = K2F_ITEMS + 1;
constexpr int K2F_MAX_LEN = 32768;

// exponent statistics of the event's float32 samples from their bit patterns: the magnitude exponent is
// that of the largest |x| (integer max of the bits), the quantum exponent is E + ctz(mantissa with its
// implicit one); zeros contribute nothing, inf/NaN poison the verdict through the magnitude.
struct K2FBits {
    unsigned amax;  // max over samples of bits(|x|)
    int elow;       // min over non-zero samples of (biased E, denormals as 1) + ctz(24-bit significand)
    __device__ __forceinline__ void init() { amax = 0u; elow = K2_ELOW_INIT; }
    __device__ __forceinline__ void add(float x)
    {
        const unsigned a = __float_as_uint(x) & 0x7fffffffu;
        amax = max(amax, a);
        const unsigned E = a >> 23;
        const unsigned sig = E ? (a | 0x00800000u) : a;       // denormal: no implicit one, exponent as for E = 1
        const int q = (int)(E ? E : 1u) + (__ffs((int)(sig & 0x00ffffffu)) - 1);
        if (a) elow = min(elow, q);
    }
    __device__ __forceinline__ void add(double) {}
};

#ifndef K2F_CFG_CTAS
#define K2F_CFG_CTAS 2
#endif
template <typename T>
__global__ void __launch_bounds__(K2F_WARPS * 32, K2F_CFG_CTAS)
k2_event_scan(PPSource src, const T *__restrict__ samples, const int64_t *__restrict__ ev_len, const PPCounters *ctr,
              unsigned *__restrict__ inexact, double2 *__restrict__ cc, int check)
{
    // per-warp staging; the input transpose (T) and the output transpose (double2) share it
    __shared__ __align__(16) double2 s_stage[K2F_WARPS][32 * K2F_PAD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double2 *sout = s_stage[warp];
    T *sin = reinterpret_cast<T *>(sout);
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t warps = (int64_t)gridDim.x * K2F_WARPS;
    // events are dealt to CTAs round-robin so that a handful of events still spreads over all SMs
    for (int64_t e = (int64_t)ctr->ev_begin + (int64_t)warp * gridDim.x + blockIdx.x; e < n_events; e += warps) {
        const int64_t len = ev_len[e];
        if (len > K2F_MAX_LEN) continue;
        const int64_t off = src.ev_off[e];
        const T *in = samples + (src.kind != PP_SRC_FLAT64 ? src.ev_start[e] : off);
        double2 *out = cc + off;
        double carry_c = 0.0, carry_c2 = 0.0;
        K2FBits fb;
        fb.init();
        K2Exp ex;   // float64 / ADC source: both x and x*x are analysed
        ex.init();
        T xv[K2F_ITEMS], xn[K2F_ITEMS];
#pragma unroll
        for (int k = 0; k < K2F_ITEMS; ++k) {
            const int q = k * 32 + lane;
            xv[k] = q < len ? __ldg(in + q) : (T)0;
        }
        for (int64_t base = 0; base < len; base += K2F_TILE) {
            const int cnt = (int)((len - base) < K2F_TILE ? (len - base) : K2F_TILE);
            // the next step's samples travel while this one is scanned
            const int64_t nb = base + K2F_TILE;
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k) {
                const int64_t q = nb + k * 32 + lane;
                xn[k] = q < len ? __ldg(in + q) : (T)0;
            }
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k) {
                const int q = k * 32 + lane;
                sin[(q / K2F_ITEMS) * K2F_PAD + (q % K2F_ITEMS)] = xv[k];
            }
            __syncwarp();
            double pc[K2F_ITEMS], pc2[K2F_ITEMS];
            double c = 0.0, c2 = 0.0;
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k) {
                const T xs = sin[lane * K2F_PAD + k];
                const double x = pp_val(xs, src.adc);
                // padding decodes to the ADC offset, which is no sample of the event: kept out of the proof
                if constexpr (sizeof(T) == 4) fb.add(xs); else if (lane * K2F_ITEMS + k < cnt) ex.add(x);
                c = __dadd_rn(c, x);
                c2 = __dadd_rn(c2, __dmul_rn(x, x));
                pc[k] = c; pc2[k] = c2;
            }
            double ic = c, ic2 = c2;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t1 = __shfl_up_sync(PP_FULL, ic, d), t2 = __shfl_up_sync(PP_FULL, ic2, d);
                if (lane >= d) { ic = __dadd_rn(t1, ic); ic2 = __dadd_rn(t2, ic2); }
            }
            __syncwarp();  // every lane has taken its inputs out of the staging area
            // exclusive prefix of this lane = carry + earlier lanes
            const double ec = __dadd_rn(carry_c, __dsub_rn(ic, c));
            const double ec2 = __dadd_rn(carry_c2, __dsub_rn(ic2, c2));
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k)
                sout[lane * K2F_PAD + k] = make_double2(__dadd_rn(ec, pc[k]), __dadd_rn(ec2, pc2[k]));
            carry_c = __dadd_rn(carry_c, __shfl_sync(PP_FULL, ic, 31));
            carry_c2 = __dadd_rn(carry_c2, __shfl_sync(PP_FULL, ic2, 31));
            __syncwarp();
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k) {
                const int q = k * 32 + lane;
                if (q < cnt) out[base + q] = sout[(q / K2F_ITEMS) * K2F_PAD + (q % K2F_ITEMS)];
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < K2F_ITEMS; ++k) xv[k] = xn[k];
        }
        if (check) {
            int el1, em1, el2, em2;
            if (sizeof(T) == 4) {
                unsigned amax = fb.amax;
                int elow = fb.elow;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    amax = max(amax, __shfl_xor_sync(PP_FULL, amax, d));
                    elow = min(elow, __shfl_xor_sync(PP_FULL, elow, d));
                }
                if (amax == 0u) { el1 = el2 = K2_ELOW_INIT; em1 = em2 = K2_EMAX_INIT; }  // all zeros: nothing to prove
                else if (amax >= 0x7f800000u) { el1 = el2 = -K2_BAD_EXP; em1 = em2 = K2_BAD_EXP; }
                else {
                    const int E = (int)(amax >> 23);
                    em1 = (E ? E : 1) - 127;          // |x| < 2^(em1 + 1)
                    el1 = elow - 127 - 23;
                    el2 = 2 * el1;                      // x*x is exact in fp64: quantum and magnitude follow from x
                    em2 = 2 * em1 + 1;
                }
            } else {
                ex.warp_reduce();
                el1 = ex.el1; em1 = ex.em1; el2 = ex.el2; em2 = ex.em2;
            }
            if (lane == 0) {
                int lg = 0;
                while ((1LL << lg) < len) ++lg;
                bool ok = true;
                if (em1 != K2_EMAX_INIT) ok = ok && ((long long)lg + em1 + 1 - el1 <= 53);
                if (em2 != K2_EMAX_INIT) ok = ok && ((long long)lg + em2 + 1 - el2 <= 53);
                inexact[e] = ok ? 0u : 1u;
            }
        }
    }
}

// exclusive prefix of tiles per event (one CTA; the event table is small)
__global__ void __launch_bounds__(1024)
k2_tile_offsets(PPCounters *ctr, const int64_t *__restrict__ ev_len, int64_t *__restrict__ ev_tile_off,
                K2EventBits *__restrict__ bits, unsigned *__restrict__ inexact)
{
    __shared__ long long wsum[32];
    __shared__ long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t ev_begin = (int64_t)ctr->ev_begin;
    const long long tiles_before = ev_begin > 0 ? (long long)ctr->n_scan_tiles : 0;
    if (tid == 0) s_carry = tiles_before;
    __syncthreads();
    for (int64_t c0 = ev_begin; c0 < n_events; c0 += 1024) {
        const int64_t e = c0 + tid;
        long long v = (e < n_events && ev_len[e] > K2F_MAX_LEN) ? (ev_len[e] + K2_TILE - 1) / K2_TILE : 0;  // short events: k2_event_scan
        long long inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            long long t = __shfl_up_sync(PP_FULL, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        long long add = 0;
        for (int w = 0; w < warp; ++w) add += wsum[w];
        const long long excl = s_carry + add + inc - v;
        if (e < n_events) {
            ev_tile_off[e] = excl;
            K2EventBits b;
            b.elow1 = b.elow2 = K2_ELOW_INIT;
            b.emax1 = b.emax2 = K2_EMAX_INIT;
            bits[e] = b;
            inexact[e] = 0u;
        }
        __syncthreads();
        if (tid == 1023) s_carry = excl + v;
        __syncthreads();
    }
    if (tid == 0) {
        ev_tile_off[n_events] = s_carry;
        ctr->n_scan_tiles = (unsigned long long)s_carry;
        ctr->tile_begin = (unsigned long long)tiles_before;
        if (ev_begin == 0) ctr->n_seq_redo = 0;
    }
}

// Which event owns `tile`, and where the tile's samples are.
struct K2Tile {
    int64_t ev, base, off;
    int cnt;
};
__device__ __forceinline__ K2Tile k2_locate(const PPSource &src, const int64_t *__restrict__ ev_len,
                                            const int64_t *__restrict__ ev_tile_off, int64_t n_events, int64_t tile)
{
    K2Tile t;
    t.ev = pp_upper_index(ev_tile_off, n_events, tile);
    t.base = (tile - ev_tile_off[t.ev]) * K2_TILE;  // sample offset inside the event
    const int64_t rest = ev_len[t.ev] - t.base;
    t.cnt = (int)(rest < K2_TILE ? rest : K2_TILE);
    t.off = src.ev_off[t.ev];
    return t;
}

// Pass 1: per-tile sums and exponent statistics.  Any summation order will do (see above).
template <typename T>
__global__ void __launch_bounds__(K2_THREADS)
k2_tile_reduce(PPSource src, const T *__restrict__ samples /* the trace, or flat for kind 1 */,
               const int64_t *__restrict__ ev_len, const int64_t *__restrict__ ev_tile_off, const PPCounters *ctr,
               K2TileState *__restrict__ tiles, K2EventBits *__restrict__ bits)
{
    __shared__ double wc[K2_THREADS / 32], wc2[K2_THREADS / 32];
    __shared__ int wex[4][K2_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t n_tiles = (int64_t)ctr->n_scan_tiles;
    for (int64_t tile = (int64_t)ctr->tile_begin + blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const K2Tile t = k2_locate(src, ev_len, ev_tile_off, n_events, tile);
        const T *in = samples + (src.kind != PP_SRC_FLAT64 ? src.ev_start[t.ev] : t.off) + t.base;
        T xv[K2_ITEMS];
#pragma unroll
        for (int i = 0; i < K2_ITEMS; ++i) {
            const int q = i * K2_THREADS + tid;
            xv[i] = q < t.cnt ? __ldg(in + q) : (T)0;
        }
        double c = 0.0, c2 = 0.0;
        K2Exp ex;
        ex.init();
#pragma unroll
        for (int i = 0; i < K2_ITEMS; ++i) {
            const double x = pp_val(xv[i], src.adc);
            if constexpr (sizeof(T) == 4) ex.add(xv[i]); else if (i * K2_THREADS + tid < t.cnt) ex.add(x);
            c = __dadd_rn(c, x);
            c2 = __dadd_rn(c2, __dmul_rn(x, x));
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            c = __dadd_rn(c, __shfl_xor_sync(PP_FULL, c, d));
            c2 = __dadd_rn(c2, __shfl_xor_sync(PP_FULL, c2, d));
        }
        ex.warp_reduce();
        __syncthreads();  // previous iteration's readers are done
        if (lane == 0) {
            wc[warp] = c; wc2[warp] = c2;
            wex[0][warp] = ex.el1; wex[1][warp] = ex.em1; wex[2][warp] = ex.el2; wex[3][warp] = ex.em2;
        }
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0, tot2 = 0.0;
            int a1 = K2_ELOW_INIT, b1 = K2_EMAX_INIT, a2 = K2_ELOW_INIT, b2 = K2_EMAX_INIT;
#pragma unroll
            for (int w = 0; w < K2_THREADS / 32; ++w) {
                tot = __dadd_rn(tot, wc[w]); tot2 = __dadd_rn(tot2, wc2[w]);
                a1 = min(a1, wex[0][w]); b1 = max(b1, wex[1][w]); a2 = min(a2, wex[2][w]); b2 = max(b2, wex[3][w]);
            }
            tiles[tile].agg_c = tot;
            tiles[tile].agg_c2 = tot2;
            if (sizeof(T) == 4 && b1 != K2_EMAX_INIT) {  // float32: x*x is exact, its exponents follow from x's
                a2 = a1 > -K2_BAD_EXP ? 2 * a1 : -K2_BAD_EXP;
                b2 = b1 < K2_BAD_EXP ? 2 * b1 + 1 : K2_BAD_EXP;
            }
            atomicMin(&bits[t.ev].elow1, a1); atomicMax(&bits[t.ev].emax1, b1);
            atomicMin(&bits[t.ev].elow2, a2); atomicMax(&bits[t.ev].emax2, b2);
        }
    }
}

// Pass 2: one warp per event -- exclusive prefix of the event's tile sums, and the exactness verdict.
__global__ void __launch_bounds__(256)
k2_event_carries(const PPCounters *ctr, const int64_t *__restrict__ ev_len, const int64_t *__restrict__ ev_tile_off,
                 K2TileState *__restrict__ tiles, const K2EventBits *__restrict__ bits, unsigned *__restrict__ inexact,
                 int check)
{
    const int lane = threadIdx.x & 31;
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = (int64_t)ctr->ev_begin + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); e < n_events;
         e += warps) {
        if (ev_len[e] <= K2F_MAX_LEN) continue;  // scanned and judged by k2_event_scan
        const int64_t t0 = ev_tile_off[e], t1 = ev_tile_off[e + 1];
        double carry_c = 0.0, carry_c2 = 0.0;
        for (int64_t b = t0; b < t1; b += 32) {
            const int64_t t = b + lane;
            const double v = t < t1 ? tiles[t].agg_c : 0.0, v2 = t < t1 ? tiles[t].agg_c2 : 0.0;
            double ic = v, ic2 = v2;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double u1 = __shfl_up_sync(PP_FULL, ic, d), u2 = __shfl_up_sync(PP_FULL, ic2, d);
                if (lane >= d) { ic = __dadd_rn(u1, ic); ic2 = __dadd_rn(u2, ic2); }
            }
            if (t < t1) {
                tiles[t].carry_c = __dadd_rn(carry_c, __dsub_rn(ic, v));
                tiles[t].carry_c2 = __dadd_rn(carry_c2, __dsub_rn(ic2, v2));
            }
            carry_c = __dadd_rn(carry_c, __shfl_sync(PP_FULL, ic, 31));
            carry_c2 = __dadd_rn(carry_c2, __shfl_sync(PP_FULL, ic2, 31));
        }
        if (check && lane == 0) {
            const long long n = ev_len[e];
            int lg = 0;
            while ((1LL << lg) < n) ++lg;
            const K2EventBits b = bits[e];
            bool ok = true;
            if (b.emax1 != K2_EMAX_INIT) ok = ok && ((long long)lg + b.emax1 + 1 - b.elow1 <= 53);
            if (b.emax2 != K2_EMAX_INIT) ok = ok && ((long long)lg + b.emax2 + 1 - b.elow2 <= 53);
            inexact[e] = ok ? 0u : 1u;
        }
    }
}

// Pass 3: per-tile scan with the carry of the earlier tiles.
template <typename T>
__global__ void __launch_bounds__(K2_THREADS, 4)
k2_tile_scan(PPSource src, const T *__restrict__ samples, const int64_t *__restrict__ ev_len,
             const int64_t *__restrict__ ev_tile_off, const PPCounters *ctr,
             const K2TileState *__restrict__ tiles, double2 *__restrict__ cc)
{
    // input staging (T) and output staging (double2) share the same shared memory
    __shared__ __align__(16) unsigned char raw[sizeof(double2) * K2_THREADS * K2_PAD];
    __shared__ double wc[K2_THREADS / 32], wc2[K2_THREADS / 32];
    T *sin = reinterpret_cast<T *>(raw);
    double2 *sout = reinterpret_cast<double2 *>(raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_events = (int64_t)ctr->n_events;
    const int64_t n_tiles = (int64_t)ctr->n_scan_tiles;

    for (int64_t tile = (int64_t)ctr->tile_begin + blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const K2Tile t = k2_locate(src, ev_len, ev_tile_off, n_events, tile);
        const T *in = samples + (src.kind != PP_SRC_FLAT64 ? src.ev_start[t.ev] : t.off) + t.base;
        const double carry_c = tiles[tile].carry_c, carry_c2 = tiles[tile].carry_c2;
        __syncthreads();  // the previous tile's output staging has been drained
        // coalesced load -> padded shared memory (conflict-free blocked reads)
#pragma unroll
        for (int i = 0; i < K2_ITEMS; ++i) {
            const int q = i * K2_THREADS + tid;
            sin[(q / K2_ITEMS) * K2_PAD + (q % K2_ITEMS)] = q < t.cnt ? __ldg(in + q) : (T)0;
        }
        __syncthreads();
        double pc[K2_ITEMS], pc2[K2_ITEMS];
        double c = 0.0, c2 = 0.0;
#pragma unroll
        for (int k = 0; k < K2_ITEMS; ++k) {
            const double x = pp_val(sin[tid * K2_PAD + k], src.adc);
            c = __dadd_rn(c, x);
            c2 = __dadd_rn(c2, __dmul_rn(x, x));
            pc[k] = c; pc2[k] = c2;
        }
        // warp scan of thread totals
        double ic = c, ic2 = c2;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double t1 = __shfl_up_sync(PP_FULL, ic, d), t2 = __shfl_up_sync(PP_FULL, ic2, d);
            if (lane >= d) { ic = __dadd_rn(t1, ic); ic2 = __dadd_rn(t2, ic2); }
        }
        if (lane == 31) { wc[warp] = ic; wc2[warp] = ic2; }
        __syncthreads();  // also: every thread has consumed its inputs from `raw`
        double wpre = carry_c, wpre2 = carry_c2;
        for (int w = 0; w < warp; ++w) { wpre = __dadd_rn(wpre, wc[w]); wpre2 = __dadd_rn(wpre2, wc2[w]); }
        // exclusive prefix of this thread = carry + earlier warps + earlier lanes
        const double ec = __dadd_rn(wpre, __dsub_rn(ic, c));
        const double ec2 = __dadd_rn(wpre2, __dsub_rn(ic2, c2));
#pragma unroll
        for (int k = 0; k < K2_ITEMS; ++k)
            sout[tid * K2_PAD + k] = make_double2(__dadd_rn(ec, pc[k]), __dadd_rn(ec2, pc2[k]));
        __syncthreads();
        double2 *dst = cc + t.off + t.base;
#pragma unroll
        for (int i = 0; i < K2_ITEMS; ++i) {
            const int q = i * K2_THREADS + tid;
            if (q < t.cnt) dst[q] = sout[(q / K2_ITEMS) * K2_PAD + (q % K2_ITEMS)];
        }
    }
}
