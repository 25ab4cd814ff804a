// split.cuh -- K3: the recursive maximum-likelihood changepoint search of
// FastStatSplit (PyPore/cparsers.pyx:26-38 var_c, :157-178 _best_split_stepwise,
// :180-203 _recursive_split) as a persistent device work queue of intervals.
//
// The recursion's result depends only on the interval [s,e) and the event's
// prefix sums (SURVEY App. A.3), so intervals can be processed in any order.
// A task is an interval of one event.  A CTA that pops a task
//   * walks the "right spine" of a long interval window by window (the
//     sequential dependency of App. A.3), scanning each window CTA-wide, pushing
//     the left child to the global queue for another CTA and continuing with
//     the right child itself; and
//   * once the interval is short enough (<= K3_CAP samples) resolves the whole
//     subtree locally, level by level: all windows of a level are cut into
//     32-candidate chunks that are spread evenly over the CTA's warps.
// Breakpoints are recorded as bits in flat event space; a compaction pass turns
// the bitmap into the sorted segment table, so no ordering is needed here.
//
// Two-stage evaluation of a window (bit-exact result, ~7x fewer instructions):
//   SCREEN  every candidate i gets an integer key
//               key(i) = n1 * L(V1) + n2 * L(V2),   L(V) = log2(V) in 2^-23 units (+ a per-window constant)
//           from a division-free variance V = Q r - (S r)^2 (r = 1/n from a table)
//           and the hardware lg2 of V's top 24 mantissa bits (MUFU.LG2), accumulated
//           exactly in 64-bit integers.  For candidates that pass the validity test
//           (V positive, normal, within 2^+-127 of the window's variance, and not
//           smaller than 2^-24 of the mean square) the distance between
//           key * ln2 / 2^23 and the reference's own fl(low + high) is rigorously
//           bounded by eps = n_window * 3.6e-7 + 1e-6  (derivation in DESIGN.md; the
//           MUFU error term is measured exhaustively by pp_debug_lg2_error).
//   EXACT   only candidates with key <= min key + 2 eps, and every window holding a
//           candidate that failed the validity test, are evaluated with the
//           reference's exact arithmetic below; the decision (strict '>' against
//           min_gain, lowest index on ties, NaN never wins) is taken on exact values
//           only.
//
// Exact arithmetic contract: every operation of var_c and of the gain is a
// separate IEEE fp64 operation in the reference's association
// (__dsub_rn/__ddiv_rn/__dmul_rn/__dadd_rn are never contracted to FMA).
#pragma once
#include "common.cuh"
#include <cooperative_groups.h>

#ifndef K3_CFG_THREADS  // development knobs: -DK3_CFG_THREADS=.. -DK3_CFG_CTAS=..
#define K3_CFG_THREADS 128
#endif
#ifndef K3_CFG_CTAS
#define K3_CFG_CTAS 7   // 72 registers; measured 6: 1.183 ms, 7: 1.097 ms (5: 1.297)
#endif
constexpr int K3_THREADS = K3_CFG_THREADS;
constexpr int K3_CTAS_PER_SM = K3_CFG_CTAS;
constexpr int K3_WARPS = K3_THREADS / 32;
constexpr int K3_CAP = 10240;   // longest interval resolved level by level inside one CTA
#ifndef K3_CFG_LIST
#define K3_CFG_LIST 128
#endif
#ifndef K3_CFG_SURE
#define K3_CFG_SURE 1
#endif
#ifndef K3_CFG_SHARE
#define K3_CFG_SHARE 0
#endif
constexpr int K3_LIST = K3_CFG_LIST;  // windows per level (more go to the global queue)
constexpr int K3_REQ = K3_CFG_LIST;   // exact-evaluation requests per level
constexpr int K3_SHARE = K3_CFG_SHARE; // both children of a split at least this long: the right one goes to the
                                       // global queue for another CTA (finer tasks, shorter tail); 0 = keep both
#ifndef K3_CFG_IDLE_SHARE
#define K3_CFG_IDLE_SHARE 512
#endif
constexpr int K3_IDLE_SHARE = K3_CFG_IDLE_SHARE;  // while CTAs are waiting for work: right children of splits whose
                                                  // halves are both at least this long go to the global queue; 0 = off.
// Only acts when the launch starts with fewer than two tasks per CTA (measured with 512: 500 events 0.252 -> 0.216 ms;
// with a full queue sharing loses: the pushes' gpu-scope fences cost more than the tail they fill).
constexpr int K3_PIECES = K3_LIST + K3_WARPS;  // (warp, window) screening records per level
// Measured on B200 at BASELINE configs[1] (profiles/r01f_k3_variants.txt): taking 2 events per CTA
// or handing intervals to idle CTAs both LOST time (the search is bound by L2 -> SM traffic of the
// prefix sums, and both widen a CTA's working set); those knobs are gone, a CTA resolves one task at a time.
#ifndef K3_CFG_LDCS
#define K3_CFG_LDCS 0
#endif
#ifndef K3_CFG_PREFETCH
#define K3_CFG_PREFETCH 1
#endif
#ifndef K3_CFG_HALFKEY
// DEVELOPMENT VARIANT, off in the product build, not yet run on a GPU (DESIGN.md 4, "planned next"): a candidate's
// screening key is L(s,i) + R(i,e) (left side, right side).  When [s,e) splits at x, the left child's candidates need
// L(s,i) + R(i,x) -- and L(s,i) is the number the parent's scan computed -- the right child's need L(x,i) + R(i,e).
// With K3_CFG_HALFKEY=1 every screened scan of the level loop stores both half-keys per flat candidate position
// (K3Global::hkL / hkR, 8 B each) and a child whose first window is its whole interval loads the inherited half
// instead of recomputing it (K3Item::pad bit 0: L valid, bit 1: R valid).  The half-keys are integers relative to the
// task's exponent base, which is constant for a task's whole local subtree; anything that leaves the CTA (global
// queue), every forced split and every window that was scanned exactly starts without inherited halves.
#define K3_CFG_HALFKEY 0
#endif
constexpr int K3_NO_EBASE = 0x7fffffff;
constexpr unsigned long long K3_NO_TICKET = ~0ull;
constexpr int K3_FULL_FLAG = 0x40000000;  // window flag: screening impossible / inconclusive / request overflow, scan exactly
constexpr int K3_MULTI_FLAG = 0x20000000; // window flag: several exact evaluations compete (two-phase argmax)
constexpr unsigned K3_ALLOC_SLOT = 1u << 20;  // level allocator: windows in the high 12 bits, 32-candidate chunks below
constexpr int K3_BAD_FLAG = 0x40000000;    // piece record: a candidate failed the validity test
constexpr int K3_RESCAN_FLAG = (int)0x80000000;  // piece record: several candidates within 2 eps of the minimum
constexpr int K3_MAX_SCREEN_W = 1 << 24;   // keys stay below 2^56

constexpr int K3_RATIO_BITS = 24;            // validity: (S/n)^2 < 2^24 * V
constexpr double K3_EPS_PER_SAMPLE = 3.6e-7; // nats; > (2^-23/ln2 + 2^-22 + 2^-24) * ln2 + 14.01 * 2^-53 * 2^24
constexpr double K3_EPS_CONST = 1e-6;
constexpr double K3_KEY_PER_NAT = 12102203.161561485;  // 2^23 / ln 2
constexpr double K3_HUGE = 1e280;
constexpr unsigned long long K3_NOKEY = ~0ull;

struct PPTask { int ev, s, e, flags; };
struct K3Item { int s, e, ps, pad; };  // interval and the start of the window to scan next
struct K3Params { int mw, MW, W; double min_gain; };
struct K3Best { double g; int x; };
struct K3Scr { unsigned long long k1, k2; int i1, bad; };  // per-lane screening state: two smallest keys
// How screened windows were decided (PPCounters::n_sure / n_multi / n_full): on the screened gain alone, by the
// argmax over several contenders' exact gains, or by an exact scan of every candidate.
struct K3Branches { unsigned sure, multi, full; };

struct K3Global {
    const double2 *cc;
    const int64_t *ev_off;
    const int64_t *ev_len;
    unsigned *bits;
    PPTask *tasks;
    int *ready;
    int64_t q_cap;
    PPCounters *ctr;
    const double *RN;  // RN[n] = 1/n for n in [1, W], RN[0] = 0
    int screen;        // 0: exact evaluation of every candidate (validation mode)
#if K3_CFG_HALFKEY
    unsigned long long *hkL, *hkR;  // half-keys per flat candidate position: n1 L(V(s,i)), n2 L(V(i,e))
#endif
};

// The windows one level of the local search scans.  A level is filled while the previous one is
// resolved: the thread that decides a window runs the bookkeeping of _recursive_split for its
// children right away (k3_place) and registers their first scannable windows here.
struct K3Level {
    K3Item item[K3_LIST];
    int c0[K3_LIST];      // first 32-candidate chunk of the window in the level's chunk space
    int cn[K3_LIST];      // chunk count (0: exact scan)
    int flag[K3_LIST];    // K3_FULL_FLAG | K3_MULTI_FLAG
};

// Per-level counters.  Three sets rotate (level mod 3): while level L is resolved its own set collects
// requests, set L+1 collects the registrations of the next level, and set L+2 -- last read right after the
// barrier that ended level L-1 -- is zeroed behind the first barrier of level L.
struct K3Count {
    unsigned alloc;       // (windows << 20) | chunks handed out so far
    int nfull;            // windows flagged K3_FULL_FLAG
    int nreq, nrescan, nmulti;
};

struct K3Shared {
    K3Level lv[2];
    K3Count cnt[3];
    unsigned long long win_thr[K3_LIST];   // min key + 2 eps
    unsigned long long best_key[K3_LIST];  // ordered key of the best exact gain (0 = none beats min_gain)
    int best_idx[K3_LIST];
    unsigned long long pc_k1[K3_PIECES];   // smallest key of the piece
    unsigned long long pc_k2[K3_PIECES];   // second smallest (== k1 on a tie)
    int pc_i1[K3_PIECES];                  // candidate index of k1 | K3_BAD_FLAG | K3_RESCAN_FLAG
    unsigned long long pc_kt[K3_PIECES];   // screening key of the window's own n log V (K3_NOKEY: not valid)
    int req_k[K3_REQ];
    int req_i[K3_REQ];
    double req_g[K3_REQ];
    double red_g[K3_WARPS];
    unsigned long long red_k[K3_WARPS];
    int red_x[K3_WARPS];
    int share;                             // right children this level may hand to CTAs that wait for work
    int few;                               // the launch started with fewer than two tasks per CTA
    int have;                              // a task was taken
    int ev;                                // current task: event, flat offset, screening exponent base
    long long off;
    int ebase;                             // biased exponent of the task's variance - 127, or K3_NO_EBASE
    PPTask task;
    unsigned long long cand, scans, exact;
    unsigned n_sure, n_multi, n_full;      // decision branches over all tasks of the CTA (PPCounters::n_sure ..)
    unsigned n_cont;                       // contenders of the window k3_cta_scan is deciding
    K3Global G;                            // copies of the kernel parameters for the out-of-line bookkeeping
    K3Params P;
};

constexpr size_t K3_SMEM_BYTES = sizeof(K3Shared);

// prefix-sum accessor: at(p) = {c[p], c2[p]} with c[-1] = c2[-1] = 0
struct K3GlobalCC {
    const double2 *g;  // event base
    __device__ __forceinline__ double2 at(int p) const
    {
        if (p < 0) return make_double2(0.0, 0.0);
        return __ldg(g + p);
    }
};

// ---------------------------------------------------------------------------
// exact path
// ---------------------------------------------------------------------------
// var_c (cparsers.pyx:31-38); start == 0 subtracts an exact 0.0, bit-identical
// to the reference's special case.
__device__ __forceinline__ double k3_var(const double2 hi, const double2 lo, int cnt)
{
    if (cnt == 0) return 0.0;
    const double n = (double)cnt;
    const double m = __ddiv_rn(__dsub_rn(hi.x, lo.x), n);
    return __dsub_rn(__ddiv_rn(__dsub_rn(hi.y, lo.y), n), __dmul_rn(m, m));
}

__device__ __forceinline__ K3Best k3_better(const K3Best a, const K3Best b)
{
    if (b.x >= 0 && (a.x < 0 || b.g > a.g || (b.g == a.g && b.x < a.x))) return b;
    return a;
}

// gain(i) of window [ps,pe) exactly as cparsers.pyx:172-174
__device__ __forceinline__ double k3_exact_gain(const double2 lo, const double2 mid, const double2 hi,
                                                int ps, int pe, int i, double tot)
{
    const double low = __dmul_rn((double)(i - ps), log(k3_var(mid, lo, i - ps)));
    const double high = __dmul_rn((double)(pe - i), log(k3_var(hi, mid, pe - i)));
    return __dsub_rn(tot, __dadd_rn(low, high));
}

__device__ __forceinline__ double k3_exact_tot(const double2 lo, const double2 hi, int ps, int pe)
{
    return __dmul_rn((double)(pe - ps), log(k3_var(hi, lo, pe - ps)));
}

// Candidates ps+mw+first, +stride, ... <= pe-mw of window [ps,pe), all exact
// (_best_split_stepwise loop, cparsers.pyx:171-177).
template <class CC>
__device__ __forceinline__ K3Best k3_scan_range(const CC &cc, int ps, int pe, int mw,
                                                double min_gain, int first, int stride)
{
    const double2 lo = cc.at(ps - 1), hi = cc.at(pe - 1);
    const double tot = k3_exact_tot(lo, hi, ps, pe);
    K3Best b;
    b.g = min_gain;
    b.x = -1;
    const int last = pe - mw;
    for (int i = ps + mw + first; i <= last; i += stride) {
        const double g = k3_exact_gain(lo, cc.at(i - 1), hi, ps, pe, i, tot);
        if (g > b.g) { b.g = g; b.x = i; }
    }
    return b;
}

__device__ __forceinline__ K3Best k3_warp_reduce(K3Best b)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        K3Best o;
        o.g = __shfl_xor_sync(PP_FULL, b.g, d);
        o.x = __shfl_xor_sync(PP_FULL, b.x, d);
        b = k3_better(b, o);
    }
    return b;
}

// CTA-wide lexicographic reduction of per-thread exact results (all threads get it)
__device__ __forceinline__ K3Best k3_cta_reduce(K3Best b, K3Shared &S)
{
    const int tid = threadIdx.x;
    b = k3_warp_reduce(b);
    __syncthreads();
    if ((tid & 31) == 0) { S.red_g[tid >> 5] = b.g; S.red_x[tid >> 5] = b.x; }
    __syncthreads();
    K3Best r;
    r.g = S.red_g[0];
    r.x = S.red_x[0];
#pragma unroll
    for (int w = 1; w < K3_WARPS; ++w) {
        K3Best o;
        o.g = S.red_g[w];
        o.x = S.red_x[w];
        r = k3_better(r, o);
    }
    return r;
}

// ---------------------------------------------------------------------------
// screening path
// ---------------------------------------------------------------------------
// Window-level screening constants.  ebase = (biased exponent of the window's own
// variance) - 127; a candidate side is valid when its variance lies within 2^+-127
// of that, so that x = exponent - ebase fits [0, 254] and L(V) fits 32 bits.
// Returns false (-> exact scan of the window) when the window variance is not a
// comfortably normal positive number.
__device__ __forceinline__ bool k3_window_ebase(double vtot, int &ebase)
{
    const int e = __double2hiint(vtot) >> 20;  // sign folded in: negative -> e < 0
    ebase = e - 127;
    return e >= 128 && e <= 1919;
}

// One side of a candidate: key += n * L(V), V = Q r - (S r)^2 with r = fl(1/n).
//   L(V) = (exponent - ebase) * 2^23 + bits(1.0f + lg2(1.mantissa[51:29]))
//        = 2^23 * (log2 V - ebase + 1150) up to the screening error.
// S and Q are the same fp64 differences the exact path forms.
__device__ __forceinline__ bool k3_side(double S, double Q, double r, unsigned n, int ebase,
                                        unsigned long long &key)
{
    const double m = __dmul_rn(S, r);
    const double m2 = __dmul_rn(m, m);
    const double V = fma(Q, r, -m2);
    const int vh = __double2hiint(V);
    const unsigned mant = (__funnelshift_l((unsigned)__double2loint(V), (unsigned)vh, 3) & 0x007fffffu) | 0x3f800000u;
    float lg;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(__uint_as_float(mant)));
    const unsigned tb = __float_as_uint(__fadd_rn(lg, 1.0f));
    const unsigned x = (unsigned)((vh >> 20) - ebase);
    const unsigned LV = x * 0x00800000u + tb;
    key += (unsigned long long)n * LV;
    // V positive/normal/in range, and (S/n)^2 < 2^24 V (hence Q/n < (2^24 + 1) V)
    return (x <= 254u) & ((__double2hiint(m2) - vh) < (K3_RATIO_BITS << 20));
}

__device__ __forceinline__ bool k3_screen_key(const double2 mid, const double r1, const double r2, const double2 lo,
                                              const double2 hi, unsigned n1, unsigned n2, int ebase,
                                              unsigned long long &key)
{
    key = 0ull;
    const bool ok1 = k3_side(__dsub_rn(mid.x, lo.x), __dsub_rn(mid.y, lo.y), r1, n1, ebase, key);
    const bool ok2 = k3_side(__dsub_rn(hi.x, mid.x), __dsub_rn(hi.y, mid.y), r2, n2, ebase, key);
    return ok1 & ok2;
}

// same, loading its operands (candidate i of window [ps,pe), i >= 1)
__device__ __forceinline__ bool k3_screen_key_at(const double2 *__restrict__ ccg, const double2 lo, const double2 hi,
                                                 int ps, int pe, int i, const double *__restrict__ RN, int ebase,
                                                 unsigned long long &key)
{
    return k3_screen_key(__ldg(ccg + (i - 1)), __ldg(RN + (i - ps)), __ldg(RN + (pe - i)), lo, hi,
                         (unsigned)(i - ps), (unsigned)(pe - i), ebase, key);
}

__device__ __forceinline__ void k3_scr_init(K3Scr &a)
{
    a.k1 = a.k2 = K3_NOKEY;
    a.i1 = -1;
    a.bad = 0;
}

__device__ __forceinline__ void k3_scr_update(K3Scr &a, bool ok, unsigned long long key, int i)
{
    if (!ok) a.bad = 1;
    else if (key < a.k2) {
        if (key < a.k1) { a.k2 = a.k1; a.k1 = key; a.i1 = i; }
        else a.k2 = key;
    }
}

#ifndef K3_CFG_UNROLL
#define K3_CFG_UNROLL 2
#endif
#ifndef K3_CFG_L1PF
#define K3_CFG_L1PF 1   // measured on configs[1] (profiles/r02c_k3_prefetch_variants.txt): k3_split 1.054 -> 1.015 ms, 2 / 3 trips no better
#endif
__device__ __forceinline__ void k3_prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#if K3_CFG_LDCS
#define K3_LD_MID(p) __ldcs(p)
#else
#define K3_LD_MID(p) __ldg(p)
#endif

// Screen candidates i, i+stride, ... <= i_last of window [ps,pe) (requires mw >= 1 so that
// n1, n2 >= 1 and i >= 1).  Plain pointer increments; two candidates per trip (four independent
// fp64 chains in flight), the operands of the next pair requested before the current one is evaluated.
__device__ __forceinline__ void k3_screen_lane(const double2 *__restrict__ ccg, const double2 lo, const double2 hi,
                                               int ps, int pe, int ebase, const double *__restrict__ RN, int i,
                                               int i_last, int stride, K3Scr &a)
{
    if (i > i_last) return;
    const double2 *pm = ccg + (i - 1);
    const double *p1 = RN + (i - ps), *p2 = RN + (pe - i);
    unsigned n1 = (unsigned)(i - ps), n2 = (unsigned)(pe - i);
#if K3_CFG_UNROLL == 2
    const int s2 = 2 * stride;
    if (i + stride <= i_last) {
        double2 mA = K3_LD_MID(pm), mB = K3_LD_MID(pm + stride);
        double rA1 = __ldg(p1), rA2 = __ldg(p2), rB1 = __ldg(p1 + stride), rB2 = __ldg(p2 - stride);
#if K3_CFG_L1PF > 0
        // the pair K3_CFG_L1PF trips ahead into L1 (no register held): the register prefetch below is issued half a
        // trip ahead at best (the compiler sinks it under the 72-register cap) and a miss to HBM takes longer
        const int pf = K3_CFG_L1PF * s2;
        if (i + pf <= i_last) k3_prefetch_l1(pm + pf);
        if (i + pf + stride <= i_last) k3_prefetch_l1(pm + pf + stride);
        if (K3_CFG_L1PF > 1) {
            if (i + s2 <= i_last) k3_prefetch_l1(pm + s2);
            if (i + s2 + stride <= i_last) k3_prefetch_l1(pm + s2 + stride);
        }
#endif
        for (;;) {
            const bool more = i + s2 + stride <= i_last;
#if K3_CFG_L1PF > 0
            if (i + pf + s2 <= i_last) k3_prefetch_l1(pm + pf + s2);
            if (i + pf + s2 + stride <= i_last) k3_prefetch_l1(pm + pf + s2 + stride);
#endif
#if !K3_CFG_PREFETCH
            if (true) {
                unsigned long long keyA, keyB;
                const bool okA = k3_screen_key(mA, rA1, rA2, lo, hi, n1, n2, ebase, keyA);
                const bool okB = k3_screen_key(mB, rB1, rB2, lo, hi, n1 + (unsigned)stride, n2 - (unsigned)stride, ebase, keyB);
                k3_scr_update(a, okA, keyA, i);
                k3_scr_update(a, okB, keyB, i + stride);
                pm += s2; p1 += s2; p2 -= s2;
                n1 += (unsigned)s2; n2 -= (unsigned)s2;
                i += s2;
                if (!more) break;
                mA = K3_LD_MID(pm); mB = K3_LD_MID(pm + stride);
                rA1 = __ldg(p1); rA2 = __ldg(p2); rB1 = __ldg(p1 + stride); rB2 = __ldg(p2 - stride);
                continue;
            }
#endif
            double2 mA_n = mA, mB_n = mB;
#if K3_CFG_PREFETCH == 2
            // only the prefix sums (L2 latency) are requested a trip ahead; the 1/n table is L1-resident
            if (more) {
                mA_n = K3_LD_MID(pm + s2);
                mB_n = K3_LD_MID(pm + s2 + stride);
            }
            unsigned long long keyA, keyB;
            const bool okA = k3_screen_key(mA, rA1, rA2, lo, hi, n1, n2, ebase, keyA);
            const bool okB = k3_screen_key(mB, rB1, rB2, lo, hi, n1 + (unsigned)stride, n2 - (unsigned)stride, ebase, keyB);
            k3_scr_update(a, okA, keyA, i);
            k3_scr_update(a, okB, keyB, i + stride);
            pm += s2; p1 += s2; p2 -= s2;
            n1 += (unsigned)s2; n2 -= (unsigned)s2;
            i += s2;
            if (!more) break;
            rA1 = __ldg(p1); rA2 = __ldg(p2); rB1 = __ldg(p1 + stride); rB2 = __ldg(p2 - stride);
            mA = mA_n; mB = mB_n;
#else
            double rA1_n = rA1, rA2_n = rA2, rB1_n = rB1, rB2_n = rB2;
            if (more) {
                mA_n = K3_LD_MID(pm + s2);
                mB_n = K3_LD_MID(pm + s2 + stride);
                rA1_n = __ldg(p1 + s2);
                rB1_n = __ldg(p1 + s2 + stride);
                rA2_n = __ldg(p2 - s2);
                rB2_n = __ldg(p2 - s2 - stride);
            }
            unsigned long long keyA, keyB;
            const bool okA = k3_screen_key(mA, rA1, rA2, lo, hi, n1, n2, ebase, keyA);
            const bool okB = k3_screen_key(mB, rB1, rB2, lo, hi, n1 + (unsigned)stride, n2 - (unsigned)stride, ebase, keyB);
            k3_scr_update(a, okA, keyA, i);
            k3_scr_update(a, okB, keyB, i + stride);
            pm += s2; p1 += s2; p2 -= s2;
            n1 += (unsigned)s2; n2 -= (unsigned)s2;
            i += s2;
            if (!more) break;
            mA = mA_n; mB = mB_n; rA1 = rA1_n; rA2 = rA2_n; rB1 = rB1_n; rB2 = rB2_n;
#endif
        }
        if (i > i_last) return;
    }
    // at most one candidate is left
    {
        unsigned long long key;
        const bool ok = k3_screen_key(K3_LD_MID(pm), __ldg(p1), __ldg(p2), lo, hi, n1, n2, ebase, key);
        k3_scr_update(a, ok, key, i);
    }
#else
    double2 mid = K3_LD_MID(pm);
    double r1 = __ldg(p1), r2 = __ldg(p2);
    for (;;) {
        const bool more = i + stride <= i_last;
        double2 mid_n = mid;
        double r1_n = r1, r2_n = r2;
        if (more) {
            mid_n = K3_LD_MID(pm + stride);
            r1_n = __ldg(p1 + stride);
            r2_n = __ldg(p2 - stride);
        }
        unsigned long long key;
        const bool ok = k3_screen_key(mid, r1, r2, lo, hi, n1, n2, ebase, key);
        k3_scr_update(a, ok, key, i);
        if (!more) break;
        mid = mid_n; r1 = r1_n; r2 = r2_n;
        pm += stride; p1 += stride; p2 -= stride;
        n1 += (unsigned)stride; n2 -= (unsigned)stride;
        i += stride;
    }
#endif
}

#if K3_CFG_HALFKEY
// k3_screen_lane with half-key reuse.  MODE 0: both sides computed and stored; 1: the left half is inherited
// (loaded), the right one computed and stored; 2: the right half is inherited.  hkL / hkR are event-based.
// Loads of half-keys written earlier in this launch by other warps of the CTA go through L2 (__ldcg / __stcg):
// the level barriers order them, the non-coherent path would not see them.
template <int MODE>
__device__ __forceinline__ void k3_hk_load(const double2 *__restrict__ ccg, const unsigned long long *hkL,
                                           const unsigned long long *hkR, const double *__restrict__ RN, int ps, int pe,
                                           int j, double2 &m, double &r1, double &r2, unsigned long long &h)
{
    m = K3_LD_MID(ccg + (j - 1));
    if (MODE != 1) r1 = __ldg(RN + (j - ps));
    if (MODE != 2) r2 = __ldg(RN + (pe - j));
    if (MODE == 1) h = __ldcg(hkL + j);
    if (MODE == 2) h = __ldcg(hkR + j);
}

template <int MODE>
__device__ __forceinline__ void k3_hk_eval(unsigned long long *hkL, unsigned long long *hkR, const double2 lo,
                                           const double2 hi, int ps, int pe, int ebase, int j, const double2 m,
                                           double r1, double r2, unsigned long long h, bool store, K3Scr &a)
{
    unsigned long long kl = 0ull, kr = 0ull;
    bool ok = true;
    if (MODE != 1) {
        ok = k3_side(__dsub_rn(m.x, lo.x), __dsub_rn(m.y, lo.y), r1, (unsigned)(j - ps), ebase, kl);
        if (store) __stcg(hkL + j, kl);
    } else {
        kl = h;
    }
    if (MODE != 2) {
        ok = ok & k3_side(__dsub_rn(hi.x, m.x), __dsub_rn(hi.y, m.y), r2, (unsigned)(pe - j), ebase, kr);
        if (store) __stcg(hkR + j, kr);
    } else {
        kr = h;
    }
    k3_scr_update(a, ok, kl + kr, j);
}

template <int MODE>
__device__ __forceinline__ void k3_screen_lane_hk(const double2 *__restrict__ ccg, unsigned long long *hkL,
                                                  unsigned long long *hkR, const double2 lo, const double2 hi, int ps,
                                                  int pe, int ebase, const double *__restrict__ RN, int i, int i_last,
                                                  int stride, bool store, K3Scr &a)
{
    // store == false: no child of this window can be scanned (leaf scans), nobody will read the halves
    if (i > i_last) return;
    // two candidates per trip; the operands of the next pair are requested before the current pair is evaluated
    double2 mA = make_double2(0.0, 0.0), mB = mA, mA_n = mA, mB_n = mA;
    double a1 = 0.0, a2 = 0.0, b1 = 0.0, b2 = 0.0, a1_n = 0.0, a2_n = 0.0, b1_n = 0.0, b2_n = 0.0;
    unsigned long long hA = 0ull, hB = 0ull, hA_n = 0ull, hB_n = 0ull;
    k3_hk_load<MODE>(ccg, hkL, hkR, RN, ps, pe, i, mA, a1, a2, hA);
    bool haveB = i + stride <= i_last;
    if (haveB) k3_hk_load<MODE>(ccg, hkL, hkR, RN, ps, pe, i + stride, mB, b1, b2, hB);
    for (;;) {
        const int in = i + 2 * stride;
        const bool nextA = haveB && in <= i_last, nextB = nextA && in + stride <= i_last;
        if (nextA) k3_hk_load<MODE>(ccg, hkL, hkR, RN, ps, pe, in, mA_n, a1_n, a2_n, hA_n);
        if (nextB) k3_hk_load<MODE>(ccg, hkL, hkR, RN, ps, pe, in + stride, mB_n, b1_n, b2_n, hB_n);
        k3_hk_eval<MODE>(hkL, hkR, lo, hi, ps, pe, ebase, i, mA, a1, a2, hA, store, a);
        if (haveB) k3_hk_eval<MODE>(hkL, hkR, lo, hi, ps, pe, ebase, i + stride, mB, b1, b2, hB, store, a);
        if (!nextA) break;
        i = in;
        mA = mA_n; a1 = a1_n; a2 = a2_n; hA = hA_n;
        mB = mB_n; b1 = b1_n; b2 = b2_n; hB = hB_n;
        haveB = nextB;
    }
}
#endif

// 2 eps of a window of n samples, in key units (rounded up)
__device__ __forceinline__ unsigned long long k3_eps2_key(int n)
{
    return (unsigned long long)(2.0 * ((double)n * K3_EPS_PER_SAMPLE + K3_EPS_CONST) * K3_KEY_PER_NAT) + 2ull;
}

// Monotone double -> u64 key (non-NaN); -0.0 is canonicalised to +0.0 first so
// that equal doubles have equal keys.
__device__ __forceinline__ unsigned long long k3_okey(double g)
{
    const long long b = __double_as_longlong(__dadd_rn(g, 0.0));
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000LL));
}

// warp-wide minimum of a 64-bit key with two 32-bit REDUX operations
__device__ __forceinline__ unsigned long long k3_warp_min_u64(unsigned long long k)
{
    const unsigned hi = (unsigned)(k >> 32);
    const unsigned mh = __reduce_min_sync(PP_FULL, hi);
    const unsigned lo = hi == mh ? (unsigned)k : 0xffffffffu;
    const unsigned ml = __reduce_min_sync(PP_FULL, lo);
    return ((unsigned long long)mh << 32) | ml;
}

// Warp-level summary of the lanes' screening states: smallest key, its candidate,
// and the second smallest key of the whole warp (== the smallest on a tie).
__device__ __forceinline__ void k3_warp_summary(const K3Scr &a, unsigned long long &K1, unsigned long long &K2,
                                                int &I1, bool &bad)
{
    const int lane = threadIdx.x & 31;
    K1 = k3_warp_min_u64(a.k1);
    const int winner = __ffs(__ballot_sync(PP_FULL, a.k1 == K1)) - 1;
    K2 = k3_warp_min_u64(lane == winner ? a.k2 : a.k1);
    I1 = __shfl_sync(PP_FULL, a.i1, winner);
    bad = __any_sync(PP_FULL, a.bad != 0);
}

// Whole CTA scans one window and returns the exact decision (spine mode).
template <class CC>
__device__ __forceinline__ K3Best k3_cta_scan(const CC &cc, int ps, int pe, const K3Params &P,
                                              const K3Global &G, K3Shared &S)
{
    const int tid = threadIdx.x;
    K3Best b;
    b.g = P.min_gain;
    b.x = -1;
    const double2 lo = cc.at(ps - 1), hi = cc.at(pe - 1);
    const double tot = k3_exact_tot(lo, hi, ps, pe);
    int ebase = 0;
    bool screen = G.screen && P.mw >= 1 && pe - ps <= K3_MAX_SCREEN_W && fabs(tot) <= K3_HUGE;
    screen = screen && k3_window_ebase(k3_var(hi, lo, pe - ps), ebase);
    K3Scr a;
    k3_scr_init(a);
    if (screen) {
        k3_screen_lane(cc.g, lo, hi, ps, pe, ebase, G.RN, ps + P.mw + tid, pe - P.mw, K3_THREADS, a);
        // a candidate that failed the validity test sends the whole window to the exact scan
        if (__syncthreads_or(a.bad)) screen = false;
    }
    if (!screen) {
        if (tid == 0 && G.screen && P.mw >= 1 && P.W <= K3_MAX_SCREEN_W) S.n_full += 1;
        b = k3_scan_range(cc, ps, pe, P.mw, P.min_gain, tid, K3_THREADS);
        return k3_cta_reduce(b, S);
    }
    unsigned long long m = k3_warp_min_u64(a.k1);
    if ((tid & 31) == 0) S.red_k[tid >> 5] = m;
    __syncthreads();
    m = S.red_k[0];
#pragma unroll
    for (int w = 1; w < K3_WARPS; ++w) m = S.red_k[w] < m ? S.red_k[w] : m;
    const unsigned long long thr = m + k3_eps2_key(pe - ps);
    // contenders of the window, summed in shared memory behind the barriers of k3_cta_reduce (no barrier of its own)
    const unsigned ncont = (a.k1 <= thr ? 1u : 0u) + (a.k2 <= thr ? 1u : 0u);
    if (ncont) atomicAdd(&S.n_cont, ncont);
    unsigned nexact = 0;
    if (a.k2 <= thr) {
        // rare: several of this thread's candidates qualify -> rescan its subset
        const int last = pe - P.mw;
        for (int i = ps + P.mw + tid; i <= last; i += K3_THREADS) {
            unsigned long long key;
            k3_screen_key_at(cc.g, lo, hi, ps, pe, i, G.RN, ebase, key);
            if (key <= thr) {
                const double g = k3_exact_gain(lo, cc.at(i - 1), hi, ps, pe, i, tot);
                ++nexact;
                if (g > b.g) { b.g = g; b.x = i; }
            }
        }
    } else if (a.k1 <= thr) {
        const double g = k3_exact_gain(lo, cc.at(a.i1 - 1), hi, ps, pe, a.i1, tot);
        ++nexact;
        if (g > b.g) { b.g = g; b.x = a.i1; }
    }
    if (nexact) atomicAdd(&S.exact, (unsigned long long)nexact);
    b = k3_cta_reduce(b, S);
    if (tid == 0) {  // every thread's contribution is in (barriers of k3_cta_reduce); reset before the next window's
        if (S.n_cont > 1) S.n_multi += 1;  // several contenders: the lowest index among equal exact gains wins
        S.n_cont = 0;
    }
    return b;
}

// ---------------------------------------------------------------------------
// bookkeeping shared by both modes
// ---------------------------------------------------------------------------
__device__ __forceinline__ void k3_emit(const K3Global &G, int64_t off, int x)
{
    const int64_t f = off + x;
    atomicOr(&G.bits[f >> 5], 1u << (unsigned)(f & 31));
}

__device__ __forceinline__ bool k3_worth(const K3Params &P, int s, int e)
{
    // an interval that can neither be scanned nor force-split is a leaf
    return ((long long)e - s > 2LL * P.mw) || (e - s > P.MW);
}

// Interval [s,e) of event ev for any CTA; its window loop resumes at ps (the windows before ps were scanned
// without a split).
__device__ void k3_push_global(const K3Global &G, int ev, int s, int e, int ps)
{
    atomicAdd((unsigned long long *)&G.ctr->q_pending, 1ull);
    const unsigned long long slot = atomicAdd(&G.ctr->q_tail, 1ull);
    if ((int64_t)slot >= G.q_cap) {
        atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE);
        atomicAdd((unsigned long long *)&G.ctr->q_pending, (unsigned long long)(-1LL));
        return;
    }
    PPTask t;
    t.ev = ev; t.s = s; t.e = e; t.flags = ps - s;
    *reinterpret_cast<int4 *>(&G.tasks[slot]) = *reinterpret_cast<int4 *>(&t);
    __threadfence();
    atomicExch(&G.ready[slot], 1);
}

__device__ __forceinline__ int k3_forced(const K3Params &P, int s, int e)
{
    const long long a = (long long)s + P.MW, b = (long long)e - P.mw;
    return (int)(a < b ? a : b);
}

__device__ __forceinline__ int k3_next_ps(const K3Params &P, int ps, int e)
{
    const long long n = (long long)ps + P.W / 2;
    return (int)(n < e ? n : e);
}

__device__ __forceinline__ int k3_window_end(const K3Params &P, const K3Item &it)
{
    const long long pe_l = (long long)it.ps + P.W;
    return (int)(pe_l < it.e ? pe_l : it.e);
}

__device__ __forceinline__ void k3_mark_full(K3Level &L, K3Count &C, int k)
{
    if (!(atomicOr(&L.flag[k], K3_FULL_FLAG) & K3_FULL_FLAG)) atomicAdd(&C.nfull, 1);
}

// The window loop of _recursive_split (cparsers.pyx:186-203) for interval `it` up to its next
// scannable window, which is registered in level `nx`; forced max_width splits on the way are
// emitted and their children handled the same way.  Run by ONE thread (many threads concurrently
// for different intervals).  A level that is full hands the interval to the global queue.
__device__ __noinline__ void k3_place(K3Shared *Sp, K3Level *nxp, K3Count *ncp, int screen, K3Item it)
{
    // the kernel parameters are read from their shared-memory copy: taking the address of the parameter structs
    // themselves would force a local-memory copy that the whole kernel then reads instead of the constant bank
    K3Shared &S = *Sp;
    const K3Global &G = S.G;
    const K3Params &P = S.P;
    K3Level &nx = *nxp;
    K3Count &nc = *ncp;
    const int mw = P.mw, MW = P.MW;
    const int64_t off = (int64_t)S.off;
    K3Item st[4];
    int sp = 0;
    for (;;) {
        // ---- one interval ----
        for (;;) {
            const long long lim = (long long)it.e - 2LL * mw;
            if (it.ps >= lim) {
                if (it.e - it.s > MW) {
                    const int x = k3_forced(P, it.s, it.e);
                    k3_emit(G, off, x);
                    K3Item l, r;
                    l.s = it.s; l.e = x; l.ps = it.s; l.pad = 0;
                    r.s = x; r.e = it.e; r.ps = x; r.pad = 0;
                    const bool wl = k3_worth(P, l.s, l.e), wr = k3_worth(P, r.s, r.e);
                    if (wl && wr) {
                        if (sp < 4) st[sp++] = r; else k3_push_global(G, S.ev, r.s, r.e, r.ps);
                        it = l;
                        continue;
                    }
                    if (wl) { it = l; continue; }
                    if (wr) { it = r; continue; }
                }
                break;
            }
            if (it.ps > (long long)it.s + MW) {
                const int x = k3_forced(P, it.s, it.e);
                k3_emit(G, off, x);  // the left part is not revisited (cparsers.pyx:189-191)
                if (!k3_worth(P, x, it.e)) break;
                it.s = x; it.ps = x;
#if K3_CFG_HALFKEY
                it.pad = 0;  // the anchor moved: nothing inherited
#endif
                continue;
            }
            const int pe = k3_window_end(P, it);
            if (pe - it.ps <= 2 * mw) { it.ps = k3_next_ps(P, it.ps, it.e); continue; }
            // a window to scan: register it
            const bool ok = screen && S.ebase != K3_NO_EBASE;
            const unsigned nch = ok ? (unsigned)((pe - it.ps - 2 * mw + 1 + 31) >> 5) : 0u;
            const unsigned old = atomicAdd(&nc.alloc, K3_ALLOC_SLOT | nch);
            const unsigned slot = old >> 20;
            if (slot >= (unsigned)K3_LIST) {
                // the level is full: another CTA continues the interval at the same window, so no window is
                // scanned twice and the work counters stay the reference's
                k3_push_global(G, S.ev, it.s, it.e, it.ps);
                break;
            }
            nx.item[slot] = it;
            nx.c0[slot] = (int)(old & (K3_ALLOC_SLOT - 1u));
            nx.cn[slot] = (int)nch;
            nx.flag[slot] = ok ? 0 : K3_FULL_FLAG;
            if (!ok) atomicAdd(&nc.nfull, 1);
            break;
        }
        if (sp == 0) break;
        it = st[--sp];
    }
}

// Apply the decision of a window scan (x = split position or -1) to its interval (cparsers.pyx:194-203).
#ifndef K3_CFG_NOINLINE_RESOLVE
#define K3_CFG_NOINLINE_RESOLVE 0  // measured: out of line 1.20 ms vs 1.15 ms inline
#endif
#if K3_CFG_NOINLINE_RESOLVE
__device__ __noinline__
#else
__device__ __forceinline__
#endif
void k3_resolve(const K3Global &G, K3Shared &S, K3Level &nx, K3Count &nc,
                                           const K3Params &P, int screen, const K3Item it, int x, int reuse = 0)
{
    // reuse (K3_CFG_HALFKEY): the window was screened and every candidate passed the validity test, i.e. its
    // half-keys are stored -- the children may inherit the half that keeps its anchor
    const int pe = k3_window_end(P, it);
    atomicAdd(&S.cand, (unsigned long long)(pe - it.ps - 2 * P.mw + 1));
    atomicAdd(&S.scans, 1ull);
    K3Item c;
    c.pad = 0;
    if (x >= 0) {
        k3_emit(G, (int64_t)S.off, x);
#if K3_CFG_HALFKEY
        c.pad = (reuse && it.ps == it.s) ? 1 : 0;
#endif
        if (k3_worth(P, it.s, x)) { c.s = it.s; c.e = x; c.ps = it.s; k3_place(&S, &nx, &nc, screen, c); }
#if K3_CFG_HALFKEY
        c.pad = (reuse && pe == it.e) ? 2 : 0;
#endif
        if (k3_worth(P, x, it.e)) {
            bool away = K3_SHARE > 0 && x - it.s >= K3_SHARE && it.e - x >= K3_SHARE;
            if (!away && K3_IDLE_SHARE > 0 && S.share > 0 && x - it.s >= K3_IDLE_SHARE && it.e - x >= K3_IDLE_SHARE)
                away = atomicSub(&S.share, 1) > 0;
            if (away) k3_push_global(G, S.ev, x, it.e, x);
            else { c.s = x; c.e = it.e; c.ps = x; k3_place(&S, &nx, &nc, screen, c); }
        }
    } else {
#if K3_CFG_HALFKEY
        c.pad = 0;
#endif
        c.s = it.s; c.e = it.e; c.ps = k3_next_ps(P, it.ps, it.e);
        k3_place(&S, &nx, &nc, screen, c);
    }
}

__device__ __forceinline__ void k3_request(K3Shared &S, K3Level &L, K3Count &C, int k, int i)
{
    const int r = atomicAdd(&C.nreq, 1);
    if (r < K3_REQ) { S.req_k[r] = k; S.req_i[r] = i; }
    else k3_mark_full(L, C, k);
}

// The (warp, window) pieces of a level: the level's chunks [0, nchunk) are dealt to
// the warps in equal contiguous shares; f(slot, first_chunk_in_window, end_chunk_in_window)
// is called for every window a warp's share touches.  Piece id = slot + warp.
template <class F>
__device__ __forceinline__ void k3_for_pieces(const K3Level &L, int warp, int nwin, int nchunk, F f)
{
    const int per = (nchunk + K3_WARPS - 1) / K3_WARPS;
    const int c_lo = warp * per;
    const int c_hi = c_lo + per < nchunk ? c_lo + per : nchunk;
    if (c_lo >= c_hi) return;
    int lo_s = 0, hi_s = nwin;  // largest slot with c0[slot] <= c_lo (the non-empty one among equals is the last)
    while (hi_s - lo_s > 1) {
        const int mid = (lo_s + hi_s) >> 1;
        if (L.c0[mid] <= c_lo) lo_s = mid; else hi_s = mid;
    }
    int slot = lo_s;
    int c = c_lo;
    while (c < c_hi) {
        while (L.c0[slot] + L.cn[slot] <= c) ++slot;
        const int w_c0 = L.c0[slot], w_c1 = w_c0 + L.cn[slot];
        const int cb = w_c1 < c_hi ? w_c1 : c_hi;
        f(slot, c - w_c0, cb - w_c0);
        c = cb;
    }
}

// Step 1 of a level: SCREEN.  Kept out of line so that the hot loop has the whole register budget to itself
// (the level loop's long-lived values are saved once per level at the call, not spilled inside the loop).
#ifndef K3_CFG_NOINLINE_SCREEN
#define K3_CFG_NOINLINE_SCREEN 0   // measured: out of line 1.33 ms vs 1.20 ms inline
#endif
#if K3_CFG_NOINLINE_SCREEN
__device__ __noinline__
#else
__device__ __forceinline__
#endif
void k3_screen_level(const K3Global &G, const K3Params &P, K3Shared &S, int cur, int nwin, int nchunk)
{
    const K3Level &L = S.lv[cur];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int mw = P.mw;
    const double2 *ccg = G.cc + S.off;
    K3GlobalCC acc;
    acc.g = ccg;
    const int ebase = S.ebase;
    k3_for_pieces(L, warp, nwin, nchunk, [&](int slot, int ca, int cb) {
        const K3Item it = L.item[slot];
        const int w_pe = k3_window_end(P, it);
        const int w_last = w_pe - mw;
        const int i_end = it.ps + mw + cb * 32 - 1;
        const double2 w_lo = acc.at(it.ps - 1), w_hi = acc.at(w_pe - 1);
        K3Scr a;
        k3_scr_init(a);
#if K3_CFG_HALFKEY
        {
            unsigned long long *hl = G.hkL + S.off, *hr = G.hkR + S.off;
            const int hmode = (it.ps == it.s && w_pe == it.e) ? (it.pad & 3) : 0;  // whole-interval windows only
            const int i0 = it.ps + mw + ca * 32 + lane, i1 = i_end < w_last ? i_end : w_last;
            // a child is at most (window - min_width) long and is scanned only if longer than 2 min_width
            const bool st = (long long)w_pe - it.ps > 3LL * mw;
            if (hmode == 1) k3_screen_lane_hk<1>(ccg, hl, hr, w_lo, w_hi, it.ps, w_pe, ebase, G.RN, i0, i1, 32, st, a);
            else if (hmode == 2) k3_screen_lane_hk<2>(ccg, hl, hr, w_lo, w_hi, it.ps, w_pe, ebase, G.RN, i0, i1, 32, st, a);
            else k3_screen_lane_hk<0>(ccg, hl, hr, w_lo, w_hi, it.ps, w_pe, ebase, G.RN, i0, i1, 32, st, a);
        }
#else
        k3_screen_lane(ccg, w_lo, w_hi, it.ps, w_pe, ebase, G.RN, it.ps + mw + ca * 32 + lane,
                       i_end < w_last ? i_end : w_last, 32, a);
#endif
        unsigned long long K1, K2;
        int I1;
        bool bad;
        k3_warp_summary(a, K1, K2, I1, bad);
        // the window's own n log V in the same fixed-point units (same error bound as a candidate side)
        unsigned long long kt = 0ull;
        const unsigned nw = (unsigned)(w_pe - it.ps);
        const bool tok = k3_side(__dsub_rn(w_hi.x, w_lo.x), __dsub_rn(w_hi.y, w_lo.y), __ldg(G.RN + nw), nw, ebase, kt);
        if (lane == 0) {
            S.pc_k1[slot + warp] = K1;
            S.pc_k2[slot + warp] = K2;
            S.pc_i1[slot + warp] = ((I1 - it.ps) & 0x1fffffff) | (bad ? K3_BAD_FLAG : 0);
            S.pc_kt[slot + warp] = tok ? kt : K3_NOKEY;
        }
    });
}

__global__ void __launch_bounds__(K3_THREADS, K3_CTAS_PER_SM) k3_split(K3Global G, K3Params P)
{
    extern __shared__ __align__(16) unsigned char k3_smem[];
    K3Shared &S = *reinterpret_cast<K3Shared *>(k3_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int mw = P.mw, MW = P.MW, W = P.W;
    const int screen = (G.screen && mw >= 1 && W <= K3_MAX_SCREEN_W) ? 1 : 0;

    if (tid == 0) {
        S.G = G;
        S.P = P;
        S.few = ((long long)G.ctr->n_events - (long long)G.ctr->ev_begin) < 2LL * gridDim.x ? 1 : 0;
        S.n_sure = 0; S.n_multi = 0; S.n_full = 0; S.n_cont = 0;
    }
    if (tid == 0 && blockIdx.x == 0) G.ctr->n_long = 0ull;  // k3_spine is done with it; ready for the next search
    for (;;) {
        __syncthreads();
        // ---- take a task -------------------------------------------------------------------
        if (tid == 0) {
            const unsigned long long h = atomicAdd(&G.ctr->q_head, 1ull);
            bool ok = false;
            for (;;) {
                if ((int64_t)h < G.q_cap && *((volatile int *)&G.ready[h]) != 0) { ok = true; break; }
                if (*((volatile long long *)&G.ctr->q_pending) <= 0) break;
                __nanosleep(256);
            }
            S.have = ok ? 1 : 0;
            if (ok) {
                __threadfence();
                const int4 t = __ldcg(reinterpret_cast<const int4 *>(&G.tasks[h]));
                PPTask tk;
                tk.ev = t.x; tk.s = t.y; tk.e = t.z; tk.flags = t.w;
                S.task = tk;
                S.ev = t.x;
                S.off = (long long)G.ev_off[t.x];
                // screening exponent base of the task: the variance of its whole interval (any value within
                // 2^+-127 of the candidates' variances will do; the validity test checks each candidate)
                K3GlobalCC a;
                a.g = G.cc + S.off;
                int ebase = 0;
                const bool eok = screen && k3_window_ebase(k3_var(a.at(tk.e - 1), a.at(tk.s - 1), tk.e - tk.s), ebase);
                S.ebase = eok ? ebase : K3_NO_EBASE;
            }
            S.share = 0;
            S.cand = 0;
            S.scans = 0;
            S.exact = 0;
            for (int q = 0; q < 3; ++q) {
                S.cnt[q].alloc = 0; S.cnt[q].nfull = 0; S.cnt[q].nreq = 0; S.cnt[q].nrescan = 0; S.cnt[q].nmulti = 0;
            }
        }
        __syncthreads();
        if (!S.have) break;

        // ---- spine mode: an interval too long to resolve locally ---------------------------------
        {
            const int ev = S.ev;
            const int64_t off = (int64_t)S.off;
            int s = S.task.s;
            const int e = S.task.e;
            K3GlobalCC acc;
            acc.g = G.cc + off;
            int ps = s + S.task.flags;  // k3_spine hands over the remainder of an event with its window position
            bool done = false;
            while ((long long)e - s > K3_CAP) {
                const long long lim = (long long)e - 2LL * mw;
                if (ps >= lim) {
                    if (e - s <= MW) { done = true; break; }
                    const int x = k3_forced(P, s, e);
                    if (tid == 0) {
                        k3_emit(G, off, x);
                        if (k3_worth(P, s, x)) k3_push_global(G, ev, s, x, s);
                    }
                    s = x; ps = s;
                    continue;
                }
                if (ps > (long long)s + MW) {
                    const int x = k3_forced(P, s, e);
                    if (tid == 0) k3_emit(G, off, x);
                    s = x; ps = s;  // the left part is not revisited (cparsers.pyx:189-191)
                    continue;
                }
                const long long pe_l = (long long)ps + W;
                const int pe = (int)(pe_l < e ? pe_l : e);
                if (pe - ps <= 2 * mw) { ps = k3_next_ps(P, ps, e); continue; }
                const K3Best b = k3_cta_scan(acc, ps, pe, P, G, S);
                if (tid == 0) {
                    atomicAdd(&S.cand, (unsigned long long)(pe - ps - 2 * mw + 1));
                    atomicAdd(&S.scans, 1ull);
                }
                if (b.x >= 0) {
                    if (tid == 0) {
                        k3_emit(G, off, b.x);
                        if (k3_worth(P, s, b.x)) k3_push_global(G, ev, s, b.x, s);
                    }
                    s = b.x; ps = s;
                } else {
                    ps = k3_next_ps(P, ps, e);
                }
            }
            if (!done && tid == 0) {
                K3Item it;
                it.s = s; it.e = e; it.ps = ps; it.pad = 0;
                k3_place(&S, &S.lv[0], &S.cnt[0], screen, it);
            }
        }

        // ---- local mode: the subtree of the task, level by level.  A level normally costs two barriers:
        //      SCREEN | barrier | DECIDE (+ resolve, which registers the next level's windows) | barrier ----
        int cur = 0, ci = 0;
        __syncthreads();  // the spine's registration into level 0
        for (;;) {
            K3Level &L = S.lv[cur], &NX = S.lv[cur ^ 1];
            K3Count &C = S.cnt[ci], &NC = S.cnt[ci == 2 ? 0 : ci + 1];
            const unsigned al = C.alloc;
            int nwin = (int)(al >> 20);
            int nchunk = (int)(al & (K3_ALLOC_SLOT - 1u));
            if (nwin == 0) break;
            if (nwin > K3_LIST) {  // the windows past the list went to the global queue; their chunks are the tail
                nwin = K3_LIST;
                nchunk = L.c0[K3_LIST - 1] + L.cn[K3_LIST - 1];
            }
            const int per = (nchunk + K3_WARPS - 1) / K3_WARPS;
            const double2 *ccg = G.cc + S.off;
            K3GlobalCC acc;
            acc.g = ccg;
            const int ebase = S.ebase;
            // CTAs waiting for work hold tickets past the queue's tail; the two loads complete behind the screening
            unsigned long long qh = 0ull, qt = 0ull;
            if (K3_IDLE_SHARE > 0 && tid == 0 && S.few) {
                qh = *((volatile unsigned long long *)&G.ctr->q_head);
                qt = *((volatile unsigned long long *)&G.ctr->q_tail);
            }
            // step 1: SCREEN -- every lane keeps the two smallest keys of its candidates of a piece
            k3_screen_level(G, P, S, cur, nwin, nchunk);
            if (K3_IDLE_SHARE > 0 && tid == 0 && S.few) {
                const long long waiting = (long long)(qh - qt);
                S.share = waiting > 0 ? (int)(waiting > 64 ? 64 : waiting) : 0;
            }
            __syncthreads();
            // step 2: DECIDE -- thread per window.  Minimum over the window's pieces; one contender within 2 eps of
            // it whose screened gain is clear of min_gain by more than the bound is decided without any exact
            // arithmetic and resolved on the spot; everything else asks for exact values.
            if (tid == 0) {  // the set level L+2 will register into; its last readers passed the barrier above
                K3Count &Z = S.cnt[ci == 0 ? 2 : ci - 1];
                Z.alloc = 0; Z.nfull = 0; Z.nreq = 0; Z.nrescan = 0; Z.nmulti = 0;
            }
            for (int k = tid; k < nwin; k += K3_THREADS) {
                const int c0 = L.c0[k], cn = L.cn[k];
                if (cn == 0) continue;  // registered for the exact scan
                const int w_first = c0 / per, w_last = (c0 + cn - 1) / per;
                unsigned long long gmin = K3_NOKEY;
                bool bad = false;
                for (int w = w_first; w <= w_last; ++w) {
                    const unsigned long long k1 = S.pc_k1[k + w];
                    gmin = k1 < gmin ? k1 : gmin;
                    bad = bad || (S.pc_i1[k + w] & K3_BAD_FLAG);
                }
                if (bad || gmin == K3_NOKEY) { k3_mark_full(L, C, k); continue; }
                const K3Item it = L.item[k];
                const int nw = k3_window_end(P, it) - it.ps;
                const unsigned long long eps2 = k3_eps2_key(nw);
                const unsigned long long thr = gmin + eps2;
                S.win_thr[k] = thr;
                int nr = 0, i_one = 0;
                bool rescan = false;
                for (int w = w_first; w <= w_last; ++w) {
                    if (S.pc_k2[k + w] <= thr) rescan = true;
                    else if (S.pc_k1[k + w] <= thr) { ++nr; i_one = it.ps + (S.pc_i1[k + w] & 0x1fffffff); }
                }
#if K3_CFG_SURE
                if (!rescan && nr == 1) {
                    // i_one is the argmax (every other candidate is more than 2 eps worse).  Its gain is
                    // tot - (low + high); screened: (kt - gmin) * ln2 / 2^23 with error <= 2 eps (+ conversions).
                    const unsigned long long kt = S.pc_kt[k + w_first];
                    if (kt != K3_NOKEY) {
                        const double d = (double)(long long)(kt - gmin);
                        const double want = P.min_gain * K3_KEY_PER_NAT;
                        const double margin = (double)eps2 + 64.0;
                        if (d > want + margin || d < want - margin) {
                            atomicAdd(&S.n_sure, 1u);
                            k3_resolve(G, S, NX, NC, P, screen, it, d > want ? i_one : -1, 1);
                            continue;
                        }
                    }
                }
#endif
                if (rescan || nr > 1) {  // several contenders: two-phase argmax over their exact gains
                    atomicOr(&L.flag[k], K3_MULTI_FLAG);
                    atomicAdd(&C.nmulti, 1);
                    S.best_key[k] = 0ull;
                    S.best_idx[k] = 0x7fffffff;
                }
                if (rescan) atomicAdd(&C.nrescan, 1);
                for (int w = w_first; w <= w_last; ++w) {
                    if (S.pc_k2[k + w] <= thr) S.pc_i1[k + w] |= K3_RESCAN_FLAG;
                    else if (S.pc_k1[k + w] <= thr) k3_request(S, L, C, k, it.ps + (S.pc_i1[k + w] & 0x1fffffff));
                }
            }
            __syncthreads();
            bool more_work = false;
            // step 2': pieces with several contenders are screened again, every contender is requested
            if (C.nrescan) {
                more_work = true;
                k3_for_pieces(L, warp, nwin, nchunk, [&](int slot, int ca, int cb) {
                    if (!(S.pc_i1[slot + warp] & K3_RESCAN_FLAG)) return;
                    if (L.flag[slot] & K3_FULL_FLAG) return;  // request list overflowed: exact scan decides
                    const K3Item it = L.item[slot];
                    const int w_pe = k3_window_end(P, it);
                    const int w_last = w_pe - mw;
                    int i_end = it.ps + mw + cb * 32 - 1;
                    i_end = i_end < w_last ? i_end : w_last;
                    const double2 w_lo = acc.at(it.ps - 1), w_hi = acc.at(w_pe - 1);
                    const unsigned long long thr = S.win_thr[slot];
                    for (int i = it.ps + mw + ca * 32 + lane; i <= i_end; i += 32) {
                        unsigned long long key;
                        k3_screen_key_at(ccg, w_lo, w_hi, it.ps, w_pe, i, G.RN, ebase, key);
                        if (key <= thr) k3_request(S, L, C, slot, i);
                    }
                });
                __syncthreads();
            }
            // step 3: EXACT evaluation of the requests, 3 lanes per request (tot / low / high).  A window with a
            // single contender is resolved on the spot.
            const int nreq = C.nreq < K3_REQ ? C.nreq : K3_REQ;
            if (nreq) {
                more_work = true;
                for (int r0 = 0; r0 < nreq; r0 += 10 * K3_WARPS) {
                    const int part = lane % 3;
                    const int r = r0 + warp * 10 + lane / 3;
                    const bool act = lane < 30 && r < nreq;
                    double v = 0.0;
                    int k = 0, i = 0, fl = 0;
                    K3Item it;
                    it.s = it.e = it.ps = it.pad = 0;
                    if (act) {
                        k = S.req_k[r];
                        i = S.req_i[r];
                        it = L.item[k];
                        fl = L.flag[k];
                        const int w_ps = it.ps, w_pe = k3_window_end(P, it);
                        const double2 lo = acc.at(w_ps - 1), hi = acc.at(w_pe - 1), mid = acc.at(i - 1);
                        if (part == 0) v = k3_exact_tot(lo, hi, w_ps, w_pe);
                        else if (part == 1) v = __dmul_rn((double)(i - w_ps), log(k3_var(mid, lo, i - w_ps)));
                        else v = __dmul_rn((double)(w_pe - i), log(k3_var(hi, mid, w_pe - i)));
                    }
                    const double low = __shfl_down_sync(PP_FULL, v, 1), high = __shfl_down_sync(PP_FULL, v, 2);
                    if (act && part == 0) {
                        const double g = __dsub_rn(v, __dadd_rn(low, high));   // cparsers.pyx:174
                        if (fl & K3_MULTI_FLAG) {
                            S.req_g[r] = g;
                            if (g > P.min_gain) atomicMax(&S.best_key[k], k3_okey(g));
                        } else if (!(fl & K3_FULL_FLAG)) {
                            k3_resolve(G, S, NX, NC, P, screen, it, g > P.min_gain ? i : -1, 1);
                        }
                    }
                }
                if (tid == 0) atomicAdd(&S.exact, (unsigned long long)nreq);
                if (C.nmulti) {
                    __syncthreads();
                    for (int r = tid; r < nreq; r += K3_THREADS) {
                        const int k = S.req_k[r];
                        if (!(L.flag[k] & K3_MULTI_FLAG)) continue;
                        const double g = S.req_g[r];
                        if (g > P.min_gain && k3_okey(g) == S.best_key[k]) atomicMin(&S.best_idx[k], S.req_i[r]);
                    }
                    __syncthreads();
                    for (int k = tid; k < nwin; k += K3_THREADS) {
                        const int fl = L.flag[k];
                        if ((fl & K3_MULTI_FLAG) && !(fl & K3_FULL_FLAG)) {
                            atomicAdd(&S.n_multi, 1u);
                            k3_resolve(G, S, NX, NC, P, screen, L.item[k], S.best_key[k] ? S.best_idx[k] : -1, 1);
                        }
                    }
                }
            }
            // step 4: windows left for the exact scan (validation mode: all of them), whole CTA each
            if (C.nfull) {
                more_work = true;
                __syncthreads();
                for (int k = 0; k < nwin; ++k) {
                    if (!(L.flag[k] & K3_FULL_FLAG)) continue;
                    const K3Item it = L.item[k];
                    const int pe = k3_window_end(P, it);
                    K3Best b = k3_scan_range(acc, it.ps, pe, mw, P.min_gain, tid, K3_THREADS);
                    b = k3_cta_reduce(b, S);
                    if (tid == 0) {
                        if (screen) {
                            atomicAdd(&S.exact, (unsigned long long)(pe - it.ps - 2 * mw + 1));
                            S.n_full += 1;
                        }
                        k3_resolve(G, S, NX, NC, P, screen, it, b.x);
                    }
                }
            }
            if (more_work) __syncthreads();  // the next level is complete
            cur ^= 1;
            ci = ci == 2 ? 0 : ci + 1;
        }
        __syncthreads();
        if (tid == 0) {
            atomicAdd(&G.ctr->n_cand, S.cand);
            atomicAdd(&G.ctr->n_scan, S.scans);
            atomicAdd(&G.ctr->n_exact, S.exact);
            atomicAdd(&G.ctr->n_tasks, 1ull);
            __threadfence();
            atomicAdd((unsigned long long *)&G.ctr->q_pending, (unsigned long long)(-1LL));
        }
    }
    if (tid == 0) {
        if (S.n_sure) atomicAdd(&G.ctr->n_sure, (unsigned long long)S.n_sure);
        if (S.n_multi) atomicAdd(&G.ctr->n_multi, (unsigned long long)S.n_multi);
        if (S.n_full) atomicAdd(&G.ctr->n_full, (unsigned long long)S.n_full);
    }
}

// ---------------------------------------------------------------------------
// Long events: the right spine of _recursive_split, one thread-block CLUSTER per event.
//
// The window loop over an interval longer than K3_CAP is sequential (the next window starts at
// the split the current one finds, SURVEY App. A.3), so its speed is the latency of ONE window
// scan -- and a scan of ~10^4 candidates is ~26 k warp instructions, i.e. issue-bound on a single
// SM.  k3_spine runs before k3_split: every event longer than K3_CAP is walked by a cluster of
// K3S_CLUSTER CTAs on as many SMs.  The cluster's threads share a window's candidates; every warp
// writes its summary (two smallest keys, argmin, validity) into the shared memory of ALL CTAs of
// the cluster (distributed shared memory), one cluster barrier makes them visible, and every thread
// of every CTA derives the same decision from them -- a single contender whose screened gain clears
// min_gain by the error bound needs no exact arithmetic.  Rank 0 records breakpoints and pushes the
// left children to the global queue; the remainder (<= K3_CAP) follows as an ordinary task with its
// window position; k3_split then resolves all of them.
// ---------------------------------------------------------------------------
#ifndef K3S_CFG_CLUSTER
#define K3S_CFG_CLUSTER 4
#endif
#ifndef K3S_CFG_THREADS
#define K3S_CFG_THREADS 512
#endif
constexpr int K3S_CLUSTER = K3S_CFG_CLUSTER;
constexpr int K3S_THREADS = K3S_CFG_THREADS;
constexpr int K3S_WARPS = K3S_THREADS / 32;
constexpr int K3S_TOTAL = K3S_CLUSTER * K3S_THREADS; // threads that share a window

struct K3SpineShared {
    // per-warp summaries of this CTA (reduced by warp 0), then per-CTA summaries of the whole cluster
    unsigned long long wk1[K3S_WARPS], wk2[K3S_WARPS];
    int wi1[K3S_WARPS];
    int wbad[K3S_WARPS];
    unsigned long long ck1[2][K3S_CLUSTER], ck2[2][K3S_CLUSTER];
    int ci1[2][K3S_CLUSTER];
    int cbad[2][K3S_CLUSTER];
    double wred_g[K3S_WARPS];
    int wred_x[K3S_WARPS];
    double cred_g[2][K3S_CLUSTER];
    int cred_x[2][K3S_CLUSTER];
    int list[K3S_THREADS];
    unsigned char flag[K3S_THREADS];
    int n_list;
};

// exact decision over per-thread partial results, cluster-wide (rare path): warps -> CTA -> cluster
__device__ __forceinline__ K3Best k3_spine_reduce(K3Best b, K3SpineShared &S, int par)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    b = k3_warp_reduce(b);
    if (lane == 0) { S.wred_g[warp] = b.g; S.wred_x[warp] = b.x; }
    __syncthreads();
    if (warp == 0) {
        K3Best c;
        c.g = lane < K3S_WARPS ? S.wred_g[lane] : 0.0;
        c.x = lane < K3S_WARPS ? S.wred_x[lane] : -1;
        c = k3_warp_reduce(c);
        if (lane == 0) {
            const int rank = (int)cluster.block_rank();
            for (int r = 0; r < K3S_CLUSTER; ++r) {
                K3SpineShared *R = cluster.map_shared_rank(&S, r);
                R->cred_g[par][rank] = c.g;
                R->cred_x[par][rank] = c.x;
            }
        }
    }
    cluster.sync();
    K3Best r;
    r.g = S.cred_g[par][0];
    r.x = S.cred_x[par][0];
#pragma unroll
    for (int w = 1; w < K3S_CLUSTER; ++w) {
        K3Best o;
        o.g = S.cred_g[par][w];
        o.x = S.cred_x[par][w];
        r = k3_better(r, o);
    }
    return r;
}

// One window [ps,pe) scanned by the whole cluster; every thread returns the same split position (or -1).
__device__ __forceinline__ int k3_spine_scan(const K3GlobalCC &acc, int ps, int pe, const K3Params &P, const K3Global &G,
                                             K3SpineShared &S, int ebase, bool screen, int par, unsigned &nexact,
                                             K3Branches &br)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = (int)cluster.block_rank();
    const int gtid = rank * K3S_THREADS + tid;
    const double2 lo = acc.at(ps - 1), hi = acc.at(pe - 1);
    // the window front only moves forward: pull the prefix sums behind the current window's end into L2 now
    // (one 128 B line per thread), so that the next windows' new samples are L2 hits instead of HBM misses
    asm volatile("prefetch.global.L2 [%0];" ::"l"(acc.g + pe + (long long)gtid * 8));
    if (screen) {
        K3Scr a;
        k3_scr_init(a);
        k3_screen_lane(acc.g, lo, hi, ps, pe, ebase, G.RN, ps + P.mw + gtid, pe - P.mw, K3S_TOTAL, a);
        unsigned long long K1, K2;
        int I1;
        bool bad;
        k3_warp_summary(a, K1, K2, I1, bad);
        unsigned long long kt = 0ull;
        const unsigned nw = (unsigned)(pe - ps);
        const bool tok = k3_side(__dsub_rn(hi.x, lo.x), __dsub_rn(hi.y, lo.y), __ldg(G.RN + nw), nw, ebase, kt);
        // warps -> CTA (warp 0, the same two-smallest summary over the warps' records) -> every CTA of the cluster
        if (lane == 0) { S.wk1[warp] = K1; S.wk2[warp] = K2; S.wi1[warp] = I1; S.wbad[warp] = bad ? 1 : 0; }
        __syncthreads();
        if (warp == 0) {
            K3Scr c;
            k3_scr_init(c);
            if (lane < K3S_WARPS) { c.k1 = S.wk1[lane]; c.k2 = S.wk2[lane]; c.i1 = S.wi1[lane]; c.bad = S.wbad[lane]; }
            unsigned long long C1, C2;
            int CI;
            bool cbad;
            k3_warp_summary(c, C1, C2, CI, cbad);
            if (lane == 0) {
                for (int r = 0; r < K3S_CLUSTER; ++r) {
                    K3SpineShared *R = cluster.map_shared_rank(&S, r);
                    R->ck1[par][rank] = C1;
                    R->ck2[par][rank] = C2;
                    R->ci1[par][rank] = CI;
                    R->cbad[par][rank] = cbad ? 1 : 0;
                }
            }
        }
        cluster.sync();
        unsigned long long gmin = K3_NOKEY;
        bool anybad = false;
#pragma unroll
        for (int w = 0; w < K3S_CLUSTER; ++w) {
            const unsigned long long k1 = S.ck1[par][w];
            gmin = k1 < gmin ? k1 : gmin;
            anybad = anybad || S.cbad[par][w];
        }
        if (!anybad && gmin != K3_NOKEY) {
            const unsigned long long eps2 = k3_eps2_key(pe - ps);
            const unsigned long long thr = gmin + eps2;
            int nr = 0, i_one = -1;
            bool rescan = false;
#pragma unroll
            for (int w = 0; w < K3S_CLUSTER; ++w) {
                if (S.ck2[par][w] <= thr) rescan = true;
                else if (S.ck1[par][w] <= thr) { ++nr; i_one = S.ci1[par][w]; }
            }
            if (!rescan && nr == 1 && tok) {
                const double d = (double)(long long)(kt - gmin);
                const double want = P.min_gain * K3_KEY_PER_NAT;
                const double margin = (double)eps2 + 64.0;
                if (d > want + margin) { ++br.sure; return i_one; }
                if (d < want - margin) { ++br.sure; return -1; }
            }
            if (rescan || nr > 1) ++br.multi;
            // contenders in the reference's exact arithmetic
            K3Best b;
            b.g = P.min_gain;
            b.x = -1;
            const double tot = k3_exact_tot(lo, hi, ps, pe);
            if (a.k2 <= thr) {
                const int last = pe - P.mw;
                for (int i = ps + P.mw + gtid; i <= last; i += K3S_TOTAL) {
                    unsigned long long key;
                    k3_screen_key_at(acc.g, lo, hi, ps, pe, i, G.RN, ebase, key);
                    if (key <= thr) {
                        const double g = k3_exact_gain(lo, acc.at(i - 1), hi, ps, pe, i, tot);
                        ++nexact;
                        if (g > b.g) { b.g = g; b.x = i; }
                    }
                }
            } else if (a.k1 <= thr) {
                const double g = k3_exact_gain(lo, acc.at(a.i1 - 1), hi, ps, pe, a.i1, tot);
                ++nexact;
                if (g > b.g) { b.g = g; b.x = a.i1; }
            }
            return k3_spine_reduce(b, S, par).x;
        }
    }
    // exact scan of every candidate (validation mode, or a candidate failed the validity test)
    if (screen) ++br.full;
    K3Best b = k3_scan_range(acc, ps, pe, P.mw, P.min_gain, gtid, K3S_TOTAL);
    if (ps + P.mw + gtid <= pe - P.mw) nexact += (unsigned)((pe - P.mw - (ps + P.mw + gtid)) / K3S_TOTAL + 1);
    return k3_spine_reduce(b, S, par).x;
}

// Queue slots of the spine kernel's leader thread.  Nothing consumes the queue before k3_spine has finished
// (k3_split is the next kernel on the stream), so a push is two plain stores into a slot reserved in bulk -- no
// fence, no atomic round trip on the window chain's critical path.  Slots left over are filled with empty tasks.
struct K3SpineQueue {
    long long next, end;
    __device__ __forceinline__ void push(const K3Global &G, int ev, int s, int e, int ps)
    {
        if (next == end) {
            next = (long long)atomicAdd(&G.ctr->q_tail, 32ull);
            atomicAdd((unsigned long long *)&G.ctr->q_pending, 32ull);
            end = next + 32;
        }
        if (next < G.q_cap) {
            PPTask t;
            t.ev = ev; t.s = s; t.e = e; t.flags = ps - s;  // the windows before ps were scanned without a split
            *reinterpret_cast<int4 *>(&G.tasks[next]) = *reinterpret_cast<int4 *>(&t);
            G.ready[next] = 1;
        } else {
            atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE);
            atomicAdd((unsigned long long *)&G.ctr->q_pending, (unsigned long long)(-1LL));
        }
        ++next;
    }
    __device__ __forceinline__ void flush(const K3Global &G, int ev)
    {
        while (next < end) push(G, ev, 0, 0, 0);
    }
};

__global__ void __cluster_dims__(K3S_CLUSTER, 1, 1) __launch_bounds__(K3S_THREADS, 1) k3_spine(K3Global G, K3Params P)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ K3SpineShared S;
    const int tid = threadIdx.x;
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / K3S_CLUSTER, ncl = gridDim.x / K3S_CLUSTER;
    const bool leader = rank == 0 && tid == 0;
    const int mw = P.mw, MW = P.MW, W = P.W;
    const bool screen_ok = G.screen && mw >= 1 && W <= K3_MAX_SCREEN_W;
    if (G.ctr->n_long == 0ull) return;  // counted by k3_init_queue: the usual case costs one load (whole cluster leaves)
    const int64_t n_events = (int64_t)G.ctr->n_events, ev_begin = (int64_t)G.ctr->ev_begin;
    int par = 0;
    K3SpineQueue Q;
    Q.next = Q.end = 0;
    // cluster c owns the long events among c, c + ncl, ...; every CTA of the cluster builds the same ordered list
    for (int64_t base = ev_begin + cid; base < n_events; base += (int64_t)K3S_THREADS * ncl) {
        __syncthreads();
        {
            const int64_t cand_ev = base + (int64_t)tid * ncl;
            bool is_long = false;
            if (cand_ev < n_events) {
                const int64_t l = G.ev_len[cand_ev];
                is_long = l > K3_CAP && l < 0x7fffffffLL;
            }
            S.flag[tid] = is_long ? 1 : 0;
        }
        __syncthreads();
        if (tid == 0) {
            int n = 0;
            for (int t = 0; t < K3S_THREADS; ++t)
                if (S.flag[t]) S.list[n++] = (int)(base + (int64_t)t * ncl);
            S.n_list = n;
        }
        __syncthreads();
        const int n_mine = S.n_list;
        for (int q = 0; q < n_mine; ++q) {
            const int ev = S.list[q];
            const int64_t off = G.ev_off[ev];
            const int e = (int)G.ev_len[ev];
            K3GlobalCC acc;
            acc.g = G.cc + off;
            // screening exponent base: the variance of the whole event (the validity test checks every candidate)
            int ebase = 0;
            const bool screen = screen_ok && k3_window_ebase(k3_var(acc.at(e - 1), acc.at(-1), e), ebase);
            int s = 0, ps = 0;
            unsigned long long cand = 0, scans = 0;
            unsigned nexact = 0;
            K3Branches br;
            br.sure = br.multi = br.full = 0u;
            while ((long long)e - s > K3_CAP) {
                const long long lim = (long long)e - 2LL * mw;
                if (ps >= lim) {
                    if (e - s <= MW) { s = e; break; }  // a leaf
                    const int x = k3_forced(P, s, e);
                    if (leader) {
                        k3_emit(G, off, x);
                        if (k3_worth(P, s, x)) Q.push(G, ev, s, x, s);
                    }
                    s = x; ps = s;
                    continue;
                }
                if (ps > (long long)s + MW) {
                    const int x = k3_forced(P, s, e);
                    if (leader) k3_emit(G, off, x);
                    s = x; ps = s;  // the left part is not revisited (cparsers.pyx:189-191)
                    continue;
                }
                const long long pe_l = (long long)ps + W;
                const int pe = (int)(pe_l < e ? pe_l : e);
                if (pe - ps <= 2 * mw) { ps = k3_next_ps(P, ps, e); continue; }
                const int x = k3_spine_scan(acc, ps, pe, P, G, S, ebase, screen, par, nexact, br);
                if (screen_ok && !screen) ++br.full;  // the event's variance rules screening out
                par ^= 1;
                cand += (unsigned long long)(pe - ps - 2 * mw + 1);
                scans += 1;
                if (x >= 0) {
                    if (leader) {
                        k3_emit(G, off, x);
                        if (k3_worth(P, s, x)) Q.push(G, ev, s, x, s);
                    }
                    s = x; ps = s;
                } else {
                    ps = k3_next_ps(P, ps, e);
                }
            }
            // the remainder is an ordinary task
            if (leader && s < e && k3_worth(P, s, e)) Q.push(G, ev, s, e, ps);
            if (leader) Q.flush(G, ev);
            // work counters: cand / scans are uniform, exact evaluations are per thread
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) nexact += __shfl_xor_sync(PP_FULL, nexact, d);
            if ((tid & 31) == 0 && nexact) atomicAdd(&G.ctr->n_exact, (unsigned long long)nexact);
            if (leader) {
                atomicAdd(&G.ctr->n_cand, cand);
                atomicAdd(&G.ctr->n_scan, scans);
                if (br.sure) atomicAdd(&G.ctr->n_sure, (unsigned long long)br.sure);
                if (br.multi) atomicAdd(&G.ctr->n_multi, (unsigned long long)br.multi);
                if (br.full) atomicAdd(&G.ctr->n_full, (unsigned long long)br.full);
            }
        }
    }
    cluster.sync();  // nobody leaves while a peer may still write into its shared memory
}

// Debug / validation: for window [ps,pe) of event `ev`, write per candidate the screened
// value (key converted to nats), the reference-arithmetic value fl(low + high) and the
// validity flag.
__global__ void __launch_bounds__(256)
k3_debug_screen(K3Global G, int ev, int ps, int pe, int mw, double *h_screen, double *h_exact,
                unsigned char *ok_out)
{
    K3GlobalCC cc;
    cc.g = G.cc + G.ev_off[ev];
    const double2 lo = cc.at(ps - 1), hi = cc.at(pe - 1);
    int ebase = 0;
    const bool wok = k3_window_ebase(k3_var(hi, lo, pe - ps), ebase);
    const int n = pe - mw - (ps + mw) + 1;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int i = ps + mw + j;
        unsigned long long key = 0;
        const bool ok = wok && k3_screen_key_at(cc.g, lo, hi, ps, pe, i, G.RN, ebase, key);
        const double2 mid = cc.at(i - 1);
        const double low = __dmul_rn((double)(i - ps), log(k3_var(mid, lo, i - ps)));
        const double high = __dmul_rn((double)(pe - i), log(k3_var(hi, mid, pe - i)));
        // key = 2^23 * sum n (log2 V - ebase + 1150)
        h_screen[j] = 0.6931471805599453094 * ((double)key / 8388608.0 + (double)(pe - ps) * (double)(ebase - 1150));
        h_exact[j] = __dadd_rn(low, high);
        ok_out[j] = ok ? 1 : 0;
    }
}

// gain(i) in the reference's exact arithmetic for every candidate i = ps+mw .. pe-mw of a batch
// of windows of one event (cparsers.pyx:224-240 _best_split_stepwise_score, :142-151
// _best_single_split).  out[out_off[w] + j] = gain of candidate ps[w]+mw+j.
__global__ void __launch_bounds__(256)
k3_window_gains(K3Global G, int ev, int n_windows, const int *__restrict__ ps_a, const int *__restrict__ pe_a, int mw,
                const int64_t *__restrict__ out_off, double *__restrict__ out)
{
    K3GlobalCC cc;
    cc.g = G.cc + G.ev_off[ev];
    for (int w = blockIdx.y; w < n_windows; w += gridDim.y) {
        const int ps = ps_a[w], pe = pe_a[w];
        const int n = pe - ps - 2 * mw + 1;
        if (n <= 0) continue;
        const double2 lo = cc.at(ps - 1), hi = cc.at(pe - 1);
        const double tot = k3_exact_tot(lo, hi, ps, pe);
        double *o = out + out_off[w];
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
            const int i = ps + mw + j;
            o[j] = k3_exact_gain(lo, cc.at(i - 1), hi, ps, pe, i, tot);
        }
    }
}

// Exhaustive measurement of the hardware term of the screening bound: over all 2^23
// float32 mantissas m in [1, 2), the largest | fixed23(1 + lg2.approx(m)) - 1 - log2(m) |
// (MUFU.LG2 error plus the rounding of the +1.0f), returned as an ordered-u64 maximum.
__global__ void __launch_bounds__(256) k3_debug_lg2_error(unsigned long long *max_bits)
{
    double worst = 0.0;
    for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < (1u << 23); k += gridDim.x * blockDim.x) {
        const float m = __uint_as_float(0x3f800000u | k);
        float lg;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(m));
        const unsigned tb = __float_as_uint(__fadd_rn(lg, 1.0f));
        const double fixed = (double)(tb - 0x3f800000u) / 8388608.0;
        const double err = fabs(fixed - log2((double)m));
        worst = err > worst ? err : worst;
    }
    atomicMax(max_bits, (unsigned long long)__double_as_longlong(worst));  // non-negative doubles order as integers
}

// RN[n] = 1/n (n = 1 .. len-1), correctly rounded; RN[0] = 0.
__global__ void __launch_bounds__(256) k3_fill_RN(double *RN, int len)
{
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < len; n += gridDim.x * blockDim.x)
        RN[n] = n > 0 ? __ddiv_rn(1.0, (double)n) : 0.0;
}

// One initial task per event of [ev_begin, n_events); event starts are segment starts.
__global__ void __launch_bounds__(256)
k3_init_queue(K3Global G, int use_spine)
{
    const int64_t n_events = (int64_t)G.ctr->n_events;
    const int64_t ev_begin = (int64_t)G.ctr->ev_begin;
    for (int64_t e = ev_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_events;
         e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = G.ev_off[e];
        const int64_t len = G.ev_len[e];
        const int64_t slot = e - ev_begin;
        atomicOr(&G.bits[off >> 5], 1u << (unsigned)(off & 31));
        if (slot < G.q_cap && len < 0x7fffffffLL) {
            PPTask t;
            t.ev = (int)e; t.s = 0; t.e = (int)len; t.flags = 0;
            if (use_spine && len > K3_CAP) {  // walked by k3_spine first; the slot keeps an empty task
                t.e = 0;
                atomicAdd(&G.ctr->n_long, 1ull);
            }
            G.tasks[slot] = t;
            G.ready[slot] = 1;
        } else {
            atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t cnt = n_events - ev_begin;
        const int64_t q = cnt < G.q_cap ? cnt : G.q_cap;
        G.ctr->q_head = 0;
        G.ctr->q_tail = (unsigned long long)q;
        G.ctr->q_pending = (long long)q;
        if (ev_begin == 0) {
            G.ctr->n_cand = 0;
            G.ctr->n_scan = 0;
            G.ctr->n_tasks = 0;
            G.ctr->n_exact = 0;
            G.ctr->n_sure = 0;
            G.ctr->n_multi = 0;
            G.ctr->n_full = 0;
        }
    }
}

// ---------------------------------------------------------------------------
// Bitmap -> sorted segment table (flat start, event id, event-relative start), for the flat range
// [ctr->flat_done, ctr->n_event_samples): the whole table in one go (flat_done = seg_done = 0), or -- streamed
// pipeline with host export -- one range per chunk, appended behind the ctr->seg_done rows already written.
// ---------------------------------------------------------------------------
constexpr int CP_THREADS = 256;
constexpr int CP_WPT = 4;                           // words per thread
constexpr int CP_BLOCK_WORDS = CP_THREADS * CP_WPT;  // 1024 words = 32768 samples

// word w of the bitmap restricted to the flat range [lo, hi)
__device__ __forceinline__ unsigned k3c_word(const unsigned *__restrict__ bits, int64_t w, int64_t lo, int64_t hi)
{
    const int64_t b0 = w << 5;
    if (b0 + 32 <= lo || b0 >= hi) return 0u;
    unsigned v = bits[w];
    if (b0 < lo) v &= ~0u << (unsigned)(lo - b0);
    if (b0 + 32 > hi) v &= ~0u >> (unsigned)(b0 + 32 - hi);
    return v;
}

__global__ void __launch_bounds__(CP_THREADS)
k3c_count(const unsigned *__restrict__ bits, const PPCounters *ctr, unsigned *__restrict__ block_count)
{
    __shared__ unsigned wsum[CP_THREADS / 32];
    const int tid = threadIdx.x;
    const int64_t lo = (int64_t)ctr->flat_done, hi = (int64_t)ctr->n_event_samples;
    const int64_t blk0 = (int64_t)blockIdx.x * CP_BLOCK_WORDS;
    if ((blk0 + CP_BLOCK_WORDS) * 32 <= lo || blk0 * 32 >= hi) return;  // outside the range: not looked at by the scan
    const int64_t w0 = blk0 + tid * CP_WPT;
    unsigned c = 0;
#pragma unroll
    for (int k = 0; k < CP_WPT; ++k) c += __popc(k3c_word(bits, w0 + k, lo, hi));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(PP_FULL, c, d);
    if ((tid & 31) == 0) wsum[tid >> 5] = c;
    __syncthreads();
    if (tid == 0) {
        unsigned t = 0;
        for (int w = 0; w < CP_THREADS / 32; ++w) t += wsum[w];
        block_count[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024)
k3c_scan(const unsigned *__restrict__ block_count, unsigned long long *__restrict__ block_off, PPCounters *ctr,
         int64_t cap_segs)
{
    __shared__ unsigned long long wtot[32];
    __shared__ unsigned long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t lo = (int64_t)ctr->flat_done, hi = (int64_t)ctr->n_event_samples;
    const int64_t b_lo = lo / (CP_BLOCK_WORDS * 32);
    const int64_t b_hi = hi > lo ? (hi - 1) / (CP_BLOCK_WORDS * 32) + 1 : b_lo;  // blocks [b_lo, b_hi) touch the range
    if (tid == 0) s_carry = ctr->seg_done;
    __syncthreads();
    for (int64_t c0 = b_lo; c0 < b_hi; c0 += 1024) {
        const int64_t b = c0 + tid;
        const unsigned long long v = b < b_hi ? block_count[b] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(PP_FULL, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        unsigned long long add = 0;
        for (int w = 0; w < warp; ++w) add += wtot[w];
        const unsigned long long excl = s_carry + add + inc - v;
        if (b < b_hi) block_off[b] = excl;
        __syncthreads();
        if (tid == 1023) s_carry = excl + v;
        __syncthreads();
    }
    if (tid == 0) {
        ctr->n_segments = s_carry;
        if ((int64_t)s_carry > cap_segs) atomicOr(&ctr->overflow, (unsigned)PP_OVF_SEGS);
    }
}

__global__ void __launch_bounds__(CP_THREADS)
k3c_write(const unsigned *__restrict__ bits, const unsigned long long *__restrict__ block_off,
          const int64_t *__restrict__ ev_off, const PPCounters *ctr, int64_t *__restrict__ seg_flat,
          int *__restrict__ seg_event, int64_t *__restrict__ seg_start, int64_t cap_segs)
{
    __shared__ unsigned wsum[CP_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t lo = (int64_t)ctr->flat_done, hi = (int64_t)ctr->n_event_samples;
    const int64_t blk0 = (int64_t)blockIdx.x * CP_BLOCK_WORDS;
    if ((blk0 + CP_BLOCK_WORDS) * 32 <= lo || blk0 * 32 >= hi) return;
    const int64_t w0 = blk0 + tid * CP_WPT;
    unsigned wv[CP_WPT];
    unsigned c = 0;
#pragma unroll
    for (int k = 0; k < CP_WPT; ++k) {
        wv[k] = k3c_word(bits, w0 + k, lo, hi);
        c += __popc(wv[k]);
    }
    unsigned inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned t = __shfl_up_sync(PP_FULL, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    unsigned add = 0;
    for (int w = 0; w < warp; ++w) add += wsum[w];
    if (c == 0) return;
    unsigned long long k = block_off[blockIdx.x] + add + inc - c;
    const int64_t n_events = (int64_t)ctr->n_events;
    int64_t ev = -1, ev_end = 0, ev_begin = 0;
#pragma unroll
    for (int q = 0; q < CP_WPT; ++q) {
        unsigned w = wv[q];
        while (w) {
            const int bit = __ffs(w) - 1;
            w &= w - 1;
            const int64_t f = (w0 + q) * 32 + bit;
            if (ev < 0) {
                ev = pp_upper_index(ev_off, n_events, f);
                ev_begin = ev_off[ev];
                ev_end = ev_off[ev + 1];
            }
            while (f >= ev_end) { ++ev; ev_begin = ev_end; ev_end = ev_off[ev + 1]; }
            if ((int64_t)k < cap_segs) {
                seg_flat[k] = f;
                seg_event[k] = (int)ev;
                seg_start[k] = f - ev_begin;
            }
            ++k;
        }
    }
}

__global__ void __launch_bounds__(256)
k3c_ends(const PPCounters *ctr, const int64_t *__restrict__ seg_flat,
         const int *__restrict__ seg_event, const int64_t *__restrict__ ev_off,
         int64_t *__restrict__ seg_end, int64_t cap_segs)
{
    int64_t S = (int64_t)ctr->n_segments;
    if (S > cap_segs) S = cap_segs;
    const int64_t total = (int64_t)ctr->n_event_samples;
    for (int64_t k = (int64_t)ctr->seg_done + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < S;
         k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t fe = (k + 1 < S) ? seg_flat[k + 1] : total;
        seg_end[k] = fe - ev_off[seg_event[k]];
    }
}

// Streamed pipeline with host export: rows [seg_done, n_segments) and events [ev_done, n_events) written straight
// into page-locked host memory (device-visible alias), coalesced per column, while the next chunk is being copied
// in the other direction.  Nothing is written (and PP_OVF_EXPORT is raised) if the host tables are too small.
struct PPHostTables {
    int64_t cap_events;
    int64_t *ev_start, *ev_len;
    int64_t cap_segments;
    int *seg_event;
    int64_t *seg_start, *seg_end;
    double *mean, *sd, *mn, *mx;
};

__global__ void __launch_bounds__(256)
k_export_tables(PPCounters *ctr, PPHostTables H, const int64_t *__restrict__ ev_start,
                const int64_t *__restrict__ ev_len, const int *__restrict__ seg_event,
                const int64_t *__restrict__ seg_start, const int64_t *__restrict__ seg_end,
                const double *__restrict__ mean, const double *__restrict__ sd, const double *__restrict__ mn,
                const double *__restrict__ mx, int with_stats)
{
    const int64_t S = (int64_t)ctr->n_segments, E = (int64_t)ctr->n_events;
    if (S > H.cap_segments || E > H.cap_events) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&ctr->overflow, (unsigned)PP_OVF_EXPORT);
        return;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t e = (int64_t)ctr->ev_done + t0; e < E; e += stride) {
        H.ev_start[e] = ev_start[e];
        H.ev_len[e] = ev_len[e];
    }
    for (int64_t k = (int64_t)ctr->seg_done + t0; k < S; k += stride) {
        H.seg_event[k] = seg_event[k];
        H.seg_start[k] = seg_start[k];
        H.seg_end[k] = seg_end[k];
        if (with_stats) {
            H.mean[k] = mean[k];
            H.sd[k] = sd[k];
            H.mn[k] = mn[k];
            H.mx[k] = mx[k];
        }
    }
}

// the next range starts where this one ended
__global__ void k_tables_advance(PPCounters *ctr)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    ctr->seg_done = ctr->n_segments;
    ctr->flat_done = ctr->n_event_samples;
    ctr->ev_done = ctr->n_events;
}
