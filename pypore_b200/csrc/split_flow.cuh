// split_flow.cuh -- K3 (flow form): the recursive changepoint search of FastStatSplit
// (PyPore/cparsers.pyx:157-203) as a persistent kernel WITHOUT level barriers.
//
// k3_split (split.cuh) resolves a task level by level: SCREEN | barrier | DECIDE | barrier.  On B200 its warps spend
// 35 % of their time waiting at those barriers (profiles/r01o_ncu_summary.csv: stall_barrier 4.5 of 13 cycles per
// issue) and the per-event serial steps bound the kernel: 512-thread CTAs are 2.6x slower than 128-thread ones
// (profiles/r02a_k3_geometry_variants.txt).  Here every WARP is an independent worker and a CTA only shares a
// work stack in shared memory:
//
//   * unit of work = a PIECE: a contiguous range of 32-candidate chunks of one window.  Windows of up to
//     K3F_MIN_PIECE chunks are one piece; larger ones are cut into at most K3F_MAXP pieces so that the warps of
//     the CTA cooperate on them.
//   * a warp pops a piece (LIFO: depth first, so a CTA keeps few windows -- and few KB of prefix sums -- live),
//     screens its candidates exactly like k3_split does (k3_screen_lane: two smallest integer keys per lane),
//     and stores the piece summary in the window record.  The warp that finishes the LAST piece of a window
//     decides it on its own -- minimum over the pieces, single contender clear of min_gain: no exact arithmetic;
//     otherwise the contenders are evaluated with the reference's arithmetic by the warp's lanes -- then runs the
//     bookkeeping of _recursive_split for the children (f_place) and pushes their pieces.
//   * all structural state (stack, free list of window records, event slots) is touched by lane 0 of a warp under
//     one CTA-level spin lock in shared memory; the critical sections are a few dozen instructions.
//   * an interval of at most K3F_LOCAL samples never reaches the shared stack: the warp that produced it resolves
//     its whole subtree on its own, depth first, from a private stack (f_local) -- no lock, no window record; the
//     bookkeeping runs uniformly in all lanes.  Nine out of ten scans of the headline workload are of this kind,
//     so the shared structures only see the top two or three levels of an event.
//   * when the stack runs dry a warp takes the next task from the global queue while its siblings finish, so a
//     CTA may hold up to K3F_EVS events at once.
//
// Results are those of k3_split bit for bit: same screening key, same error bound, same exact arithmetic, same
// transition function; only the order in which windows are visited differs, and the result of a window depends
// on nothing but its interval and the event's prefix sums (SURVEY App. A.3).  Every split test runs both kernels.
//
// STATUS (B200, profiles/r02b_*, r02c_*): correct on the whole parity suite and the full-size fixtures, and NOT
// faster -- 1.06..1.08 ms against k3_split's 1.02..1.05 ms on BASELINE configs[1], slower with few events (C1:
// 0.29 vs 0.22 ms).  Without barriers the warps stall on the prefix-sum loads instead (long_scoreboard 3.5 cycles
// per issue, 19 % of all samples on the first use of the pair prefetched half a trip earlier); both kernels end at
// the same ~0.6 instructions per cycle and scheduler.  k3_split therefore stays the default
// (PP_OPT_SPLIT_KERNEL = 1 selects this kernel).
#pragma once
#include "split.cuh"

#ifndef K3F_CFG_CTAS
#define K3F_CFG_CTAS 7
#endif
#ifndef K3F_CFG_MIN_PIECE
#define K3F_CFG_MIN_PIECE 32
#endif
#ifndef K3F_CFG_MAXP
#define K3F_CFG_MAXP 8
#endif
#ifndef K3F_CFG_THREADS
#define K3F_CFG_THREADS 128
#endif
constexpr int K3F_THREADS = K3F_CFG_THREADS;
constexpr int K3F_WARPS = K3F_THREADS / 32;
constexpr int K3F_CTAS_PER_SM = K3F_CFG_CTAS;
constexpr int K3F_MAXP = K3F_CFG_MAXP;            // pieces per window (<= 16: a stack entry packs the piece in 4 bits)
constexpr int K3F_MIN_PIECE = K3F_CFG_MIN_PIECE;  // chunks; a window of at most this many chunks is one piece
constexpr int K3F_WINS = 48;                      // window records per CTA
constexpr int K3F_STACK = K3F_WINS * K3F_MAXP;
#ifndef K3F_CFG_EVS
#define K3F_CFG_EVS 3
#endif
// Events in flight per CTA.  A warp that finds the shared stack empty takes the next task of the global queue, so
// that the decide / hand-out gaps of one event are filled with the scans of another -- but no more than this many:
// with 8 slots the first CTAs to start drained the whole queue (5000 events, 1036 CTAs) and the rest of the grid
// idled (measured: 1.25 ms, a third of all instructions spent polling).
constexpr int K3F_EVS = K3F_CFG_EVS;
#ifndef K3F_CFG_LOCAL
#define K3F_CFG_LOCAL 2048
#endif
constexpr int K3F_LOCAL = K3F_CFG_LOCAL;          // intervals up to this many samples: resolved by one warp, privately
constexpr int K3F_LSTACK = 24;                    // private stack entries per warp (overflow goes to the shared stack)
#ifndef PP_SPLIT_KERNEL_DEFAULT
#define PP_SPLIT_KERNEL_DEFAULT 0
#endif
constexpr long long K3F_SPIN_LIMIT = 1LL << 26;   // safety net for the waits (a broken queue must not hang the GPU)

struct K3FWin {
    int s, e, ps;            // interval and the start of the window being scanned
    short evs;               // event slot
    unsigned char npieces;
    unsigned char exact;     // pieces are scanned with the reference's arithmetic (screening impossible / switched off)
    int piece_chunks;
    int done;                // finished pieces
    int pad;
    unsigned long long k1[K3F_MAXP];   // screened: smallest key of the piece; exact: bits of its best gain
    unsigned long long k2[K3F_MAXP];   // screened: second smallest key
    int i1[K3F_MAXP];                  // candidate of k1 (| K3_BAD_FLAG); exact: best split position or -1
};

struct K3FEvent {
    long long off;
    int ev;      // -1: slot is free
    int ebase;
    int live;    // windows registered and not yet resolved (+1 while an interval is being placed)
    int pad;
};

struct K3FShared {
    K3FWin win[K3F_WINS];
    int free_list[K3F_WINS];
    int stack[K3F_STACK];
    K3FEvent evs[K3F_EVS];
    K3Item lst[K3F_WARPS][K3F_LSTACK];   // private stacks of the warps
    int n_free, top, lock, fetching, drained, few, failed, pad;
    unsigned long long cand, scans, exact, tasks;
    unsigned long long sure, multi, full;   // decision branches (PPCounters::n_sure ..)
    K3Global G;
    K3Params P;
};

constexpr size_t K3F_SMEM_BYTES = sizeof(K3FShared);

__device__ __forceinline__ void f_lock(K3FShared &S)
{
    while (atomicCAS(&S.lock, 0, 1) != 0) { }
    __threadfence_block();
}

__device__ __forceinline__ void f_unlock(K3FShared &S)
{
    __threadfence_block();
    atomicExch(&S.lock, 0);
}

__device__ __forceinline__ void f_push_global(const K3Global &G, int ev, int s, int e, int ps)
{
    atomicAdd((unsigned long long *)&G.ctr->q_pending, 1ull);
    const unsigned long long slot = atomicAdd(&G.ctr->q_tail, 1ull);
    if ((int64_t)slot >= G.q_cap) {
        atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE);
        atomicAdd((unsigned long long *)&G.ctr->q_pending, (unsigned long long)(-1LL));
        return;
    }
    PPTask t;
    t.ev = ev; t.s = s; t.e = e; t.flags = ps - s;  // the windows before ps were scanned without a split
    *reinterpret_cast<int4 *>(&G.tasks[slot]) = *reinterpret_cast<int4 *>(&t);
    __threadfence();
    atomicExch(&G.ready[slot], 1);
}

// An event slot lost its last live window: the task is finished.
__device__ __forceinline__ void f_finish_event(K3FShared &S, int es)
{
    S.evs[es].ev = -1;
    S.tasks += 1;
    __threadfence();
    atomicAdd((unsigned long long *)&S.G.ctr->q_pending, (unsigned long long)(-1LL));
}

// Register window [it.ps, min(it.e, it.ps + W)) of interval `it` and push its pieces.  Lane 0, lock held.
__device__ __forceinline__ void f_register(K3FShared &S, int es, const K3Item &it, int screen)
{
    const K3Params &P = S.P;
    const int pe = k3_window_end(P, it);
    const int nch = (pe - it.ps - 2 * P.mw + 1 + 31) >> 5;
    if (S.n_free == 0) {
        f_push_global(S.G, S.evs[es].ev, it.s, it.e, it.ps);   // another CTA (or this one, later) continues it
        return;
    }
    const int w = S.free_list[--S.n_free];
    K3FWin &Wn = S.win[w];
    int np = 1, pc = nch;
    if (nch > K3F_MIN_PIECE) {
        np = (nch + K3F_MIN_PIECE - 1) / K3F_MIN_PIECE;
        if (np > K3F_MAXP) np = K3F_MAXP;
        pc = (nch + np - 1) / np;
        np = (nch + pc - 1) / pc;
    }
    Wn.s = it.s; Wn.e = it.e; Wn.ps = it.ps;
    Wn.evs = (short)es;
    Wn.npieces = (unsigned char)np;
    Wn.exact = (screen && S.evs[es].ebase != K3_NO_EBASE) ? 0 : 1;
    Wn.piece_chunks = pc;
    Wn.done = 0;
    S.evs[es].live += 1;
    for (int p = np - 1; p >= 0; --p) S.stack[S.top++] = (w << 4) | p;
}

// The window loop of _recursive_split (cparsers.pyx:186-203) for interval `it` up to its next scannable window,
// which is registered; forced max_width splits on the way are emitted and their children handled the same way.
// Lane 0, lock held.
__device__ __noinline__ void f_place(K3FShared *Sp, int es, int screen, K3Item it)
{
    K3FShared &S = *Sp;
    const K3Global &G = S.G;
    const K3Params &P = S.P;
    const int mw = P.mw, MW = P.MW;
    const int64_t off = (int64_t)S.evs[es].off;
    K3Item st[4];
    int sp = 0;
    for (;;) {
        for (;;) {  // one interval
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
                        if (sp < 4) st[sp++] = r; else f_push_global(G, S.evs[es].ev, r.s, r.e, r.s);
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
                continue;
            }
            const int pe = k3_window_end(P, it);
            if (pe - it.ps <= 2 * mw) { it.ps = k3_next_ps(P, it.ps, it.e); continue; }
            f_register(S, es, it, screen);
            break;
        }
        if (sp == 0) break;
        it = st[--sp];
    }
}

// ---------------------------------------------------------------------------------------------------
// scanning and deciding (whole warp, uniform results).  The rarely taken paths are out of line so that the loop
// a warp lives in stays small (the first cut of this kernel stalled 2.3 cycles per issue on instruction fetch).
// ---------------------------------------------------------------------------------------------------
// candidates i0, i0 + 32, ... <= i_end of window [ps,pe) in the reference's arithmetic (_best_split_stepwise,
// cparsers.pyx:171-177): best gain above min_gain and its candidate, or (min_gain, -1); warp-uniform
__device__ __noinline__ K3Best f_exact_range(const double2 *ccg, int ps, int pe, int i0, int i_end, double min_gain)
{
    K3GlobalCC acc;
    acc.g = ccg;
    const double2 lo = acc.at(ps - 1), hi = acc.at(pe - 1);
    const double tot = k3_exact_tot(lo, hi, ps, pe);
    K3Best b;
    b.g = min_gain;
    b.x = -1;
    for (int i = i0; i <= i_end; i += 32) {
        const double g = k3_exact_gain(lo, acc.at(i - 1), hi, ps, pe, i, tot);
        if (g > b.g) { b.g = g; b.x = i; }
    }
    return k3_warp_reduce(b);
}

// one candidate in the reference's arithmetic: does it beat min_gain?
__device__ __noinline__ bool f_exact_one(const double2 *ccg, int ps, int pe, int i, double min_gain)
{
    K3GlobalCC acc;
    acc.g = ccg;
    const double2 lo = acc.at(ps - 1), hi = acc.at(pe - 1);
    return k3_exact_gain(lo, acc.at(i - 1), hi, ps, pe, i, k3_exact_tot(lo, hi, ps, pe)) > min_gain;
}

// several contenders within 2 eps of the smallest key: their exact gains, largest wins, lowest index on ties.
// `single` / `rescan`: pieces with one contender (lane p holds its candidate in I1) / with several (screened again)
__device__ __noinline__ int f_contend(const double *RN, const double2 *ccg, int ps, int pe, int mw, int ebase, int pc,
                                      double min_gain, unsigned long long thr, unsigned single, unsigned rescan, int I1,
                                      unsigned &nexact)
{
    const int lane = threadIdx.x & 31;
    K3GlobalCC acc;
    acc.g = ccg;
    const double2 lo = acc.at(ps - 1), hi = acc.at(pe - 1);
    const double tot = k3_exact_tot(lo, hi, ps, pe);
    K3Best b;
    b.g = min_gain;
    b.x = -1;
    unsigned cnt = 0;
    if (single & (1u << lane)) {
        const int i = ps + (I1 & 0x1fffffff);
        const double g = k3_exact_gain(lo, acc.at(i - 1), hi, ps, pe, i, tot);
        ++cnt;
        if (g > b.g) { b.g = g; b.x = i; }
    }
    const int w_last = pe - mw;
    for (unsigned m = rescan; m; m &= m - 1) {
        const int p = __ffs(m) - 1;
        int i_end = ps + mw + (p + 1) * pc * 32 - 1;
        i_end = i_end < w_last ? i_end : w_last;
        K3Best r;
        r.g = min_gain;
        r.x = -1;
        for (int i = ps + mw + p * pc * 32 + lane; i <= i_end; i += 32) {
            unsigned long long key;
            k3_screen_key_at(ccg, lo, hi, ps, pe, i, RN, ebase, key);
            if (key <= thr) {
                const double g = k3_exact_gain(lo, acc.at(i - 1), hi, ps, pe, i, tot);
                ++cnt;
                if (g > r.g) { r.g = g; r.x = i; }
            }
        }
        b = k3_better(b, r);
    }
    b = k3_warp_reduce(b);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(PP_FULL, cnt, d);
    nexact += cnt;
    return b.x;
}

// Decide a screened window from its pieces' summaries: split position or -1.  K1 / K2 / I1 hold, in lane p < np,
// the summary of piece p (other lanes: K3_NOKEY / -1); pc = chunks per piece.
__device__ __forceinline__ int f_decide(const K3Global &G, const K3Params &P, const double2 *ccg, const double2 lo,
                                        const double2 hi, int ps, int pe, int ebase, int np, int pc,
                                        unsigned long long K1, unsigned long long K2, int I1, unsigned &nexact,
                                        K3Branches &br)
{
    const int lane = threadIdx.x & 31;
    const int mw = P.mw;
    const bool anybad = __any_sync(PP_FULL, lane < np && (I1 & K3_BAD_FLAG));
    const unsigned long long gmin = k3_warp_min_u64(K1);
    if (anybad || gmin == K3_NOKEY) {
        // a candidate failed the validity test: the whole window in the reference's arithmetic
        nexact += (unsigned)(pe - ps - 2 * mw + 1);
        ++br.full;
        return f_exact_range(ccg, ps, pe, ps + mw + lane, pe - mw, P.min_gain).x;
    }
    const unsigned long long eps2 = k3_eps2_key(pe - ps);
    const unsigned long long thr = gmin + eps2;
    const unsigned rescan = __ballot_sync(PP_FULL, lane < np && K2 <= thr);
    const unsigned single = __ballot_sync(PP_FULL, lane < np && K2 > thr && K1 <= thr);
    if (rescan || __popc(single) != 1) {
        ++br.multi;
        return f_contend(G.RN, ccg, ps, pe, mw, ebase, pc, P.min_gain, thr, single, rescan, I1, nexact);
    }
    const int i_one = ps + (__shfl_sync(PP_FULL, I1, __ffs(single) - 1) & 0x1fffffff);
    unsigned long long kt = 0ull;
    const unsigned nw = (unsigned)(pe - ps);
    if (k3_side(__dsub_rn(hi.x, lo.x), __dsub_rn(hi.y, lo.y), __ldg(G.RN + nw), nw, ebase, kt)) {
        // i_one is the argmax (every other candidate is more than 2 eps worse); its screened gain
        // (kt - gmin) ln2 / 2^23 is within 2 eps (+ conversions) of the reference's
        const double d = (double)(long long)(kt - gmin);
        const double want = P.min_gain * K3_KEY_PER_NAT;
        const double margin = (double)eps2 + 64.0;
        if (d > want + margin) { ++br.sure; return i_one; }
        if (d < want - margin) { ++br.sure; return -1; }
    }
    nexact += 1;
    return f_exact_one(ccg, ps, pe, i_one, P.min_gain) ? i_one : -1;
}

struct K3FTally { unsigned long long cand, scans, exact; K3Branches br; };   // per warp, in registers; lane 0's copy counts

// Take the next task of the global queue.  Lane 0 acts, no lock held; returns (event slot << 8 | 1) when the task's
// interval went onto the calling warp's private stack, -1 otherwise (placed on the shared stack, empty, or none left).
__device__ __noinline__ int f_fetch(K3FShared *Sp, int screen)
{
    K3FShared &S = *Sp;
    const K3Global &G = S.G;
    const unsigned long long h = atomicAdd(&G.ctr->q_head, 1ull);
    bool ok = false;
    for (long long spin = 0;; ++spin) {
        if ((int64_t)h < G.q_cap && *((volatile int *)&G.ready[h]) != 0) { ok = true; break; }
        if (*((volatile long long *)&G.ctr->q_pending) <= 0) break;
        if (spin > (K3F_SPIN_LIMIT >> 4)) { atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE); S.failed = 1; break; }
        __nanosleep(1000);
    }
    if (!ok) {
        f_lock(S);
        S.drained = 1;
        S.fetching = 0;
        f_unlock(S);
        return -1;
    }
    __threadfence();
    const int4 t = __ldcg(reinterpret_cast<const int4 *>(&G.tasks[h]));
    const long long off = (long long)G.ev_off[t.x];
    // screening exponent base of the task: the variance of its whole interval (any value within 2^+-127 of the
    // candidates' variances will do; the validity test checks each candidate)
    int ebase = K3_NO_EBASE;
    if (t.z > t.y) {
        K3GlobalCC a;
        a.g = G.cc + off;
        int eb = 0;
        if (screen && k3_window_ebase(k3_var(a.at(t.z - 1), a.at(t.y - 1), t.z - t.y), eb)) ebase = eb;
    }
    f_lock(S);
    int es = 0;
    while (es < K3F_EVS - 1 && S.evs[es].ev >= 0) ++es;   // a slot is free: the fetch was granted on that condition
    S.evs[es].ev = t.x;
    S.evs[es].off = off;
    S.evs[es].ebase = ebase;
    S.evs[es].live = 1;    // this warp's hold on the slot
    S.fetching = 0;
    int r = -1;
    if (k3_worth(S.P, t.y, t.z)) {
        K3Item it;
        it.s = t.y; it.e = t.z; it.ps = t.y + t.w; it.pad = 0;  // k3_spine hands over a remainder with its window position
        if (it.e - it.s <= K3F_LOCAL) {
            S.lst[threadIdx.x >> 5][0] = it;
            r = (es << 8) | 1;
        } else {
            f_place(&S, es, screen, it);
        }
    }
    if (r < 0 && --S.evs[es].live == 0) f_finish_event(S, es);
    f_unlock(S);
    return r;
}

// A window of a shared record is decided (lane 0): its big children go onto the shared stack, the record is freed.
// `keeps` = small children already sit on the calling warp's private stack: the window's hold on the event slot
// passes to the warp.  One lock round trip.
__device__ __noinline__ void f_retire(K3FShared *Sp, int es, int screen, int w, const K3Item *kids, int nk, int keeps)
{
    K3FShared &S = *Sp;
    f_lock(S);
    for (int k = 0; k < nk; ++k) f_place(&S, es, screen, kids[k]);
    S.free_list[S.n_free++] = w;
    if (!keeps && --S.evs[es].live == 0) f_finish_event(S, es);
    f_unlock(S);
}

__global__ void __launch_bounds__(K3F_THREADS, K3F_CTAS_PER_SM) k3_flow(K3Global G, K3Params P)
{
    extern __shared__ __align__(16) unsigned char k3f_smem[];
    K3FShared &S = *reinterpret_cast<K3FShared *>(k3f_smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int mw = P.mw, MW = P.MW;
    const int screen = (G.screen && mw >= 1 && P.W <= K3_MAX_SCREEN_W) ? 1 : 0;
    K3Item *st = S.lst[tid >> 5];   // this warp's private stack

    if (tid == 0) {
        S.G = G;
        S.P = P;
        S.few = ((long long)G.ctr->n_events - (long long)G.ctr->ev_begin) < 2LL * gridDim.x ? 1 : 0;
        S.n_free = K3F_WINS;
        S.top = 0; S.lock = 0; S.fetching = 0; S.drained = 0; S.failed = 0;
        S.cand = S.scans = S.exact = S.tasks = 0ull;
        S.sure = S.multi = S.full = 0ull;
        for (int e = 0; e < K3F_EVS; ++e) { S.evs[e].ev = -1; S.evs[e].live = 0; }
    }
    for (int k = tid; k < K3F_WINS; k += K3F_THREADS) S.free_list[k] = K3F_WINS - 1 - k;
    if (tid == 0 && blockIdx.x == 0) G.ctr->n_long = 0ull;  // k3_spine is done with it; ready for the next search
    __syncthreads();

    K3FTally T;
    T.cand = T.scans = T.exact = 0ull;
    T.br.sure = T.br.multi = T.br.full = 0u;
    long long idle = 0;
    int ln = 0;     // entries on the private stack (all of event slot `les`)
    int les = -1;   // event slot this warp holds one `live` count of (while it has, or just had, private work)
    for (;;) {
        K3Item it;
        int es, w = -1, p = 0, np = 1, pc = 0;
        bool exact;
        if (ln > 0) {
            // ---- private work first: depth first, no lock ---------------------------------------------
            it = st[--ln];
            __syncwarp();   // everybody has read the entry before lane 0 may overwrite it
            es = les;
        } else {
            // ---- the CTA's shared stack, else the global queue ------------------------------------------
            int action = 0, entry = 0;   // 0: nothing right now, 1: a piece, 2: a private subtree, 3: leave, 5: look again
            if (lane == 0 && (idle == 0 || les >= 0 || *((volatile int *)&S.top) > 0 || (idle & 7) == 0)) {   // (a waiting warp
                // polls the stack height without the lock and looks at everything else every eighth time)
                f_lock(S);
                if (les >= 0 && --S.evs[les].live == 0) f_finish_event(S, les);   // the private work of that event is done
                if (S.top > 0) {
                    entry = S.stack[--S.top];
                    action = 1;
                } else if (S.failed) {
                    action = 3;
                } else {
                    int free_ev = 0;
                    for (int e = 0; e < K3F_EVS; ++e) free_ev += S.evs[e].ev < 0;
                    if (S.drained) action = (free_ev == K3F_EVS && !S.fetching) ? 3 : 0;
                    else if (!S.fetching && free_ev > 0 && S.n_free >= 4) { S.fetching = 1; action = 4; }
                }
                f_unlock(S);
                if (action == 4) {   // the next task of the global queue
                    entry = f_fetch(&S, screen);
                    action = entry >= 0 ? 2 : 5;
                }
            }
            les = -1;
            action = __shfl_sync(PP_FULL, action, 0);
            entry = __shfl_sync(PP_FULL, entry, 0);
            if (action == 3) break;
            if (action == 0) {
                if (++idle > (K3F_SPIN_LIMIT >> 3)) {   // never expected: leave instead of hanging the device
                    if (lane == 0) { atomicOr(&G.ctr->overflow, (unsigned)PP_OVF_QUEUE); S.failed = 1; }
                    break;
                }
                __nanosleep(500);
                continue;
            }
            idle = 0;
            if (action == 5) continue;
            if (action == 2) {   // a task's root interval sits on the private stack
                les = entry >> 8;
                ln = 1;
                continue;
            }
            w = entry >> 4;
            p = entry & 15;
            const K3FWin &Wn = S.win[w];
            it.s = Wn.s; it.e = Wn.e; it.ps = Wn.ps; it.pad = 0;
            es = Wn.evs;
            np = Wn.npieces;
            pc = Wn.piece_chunks;
        }
        const long long off = S.evs[es].off;
        const int ebase = S.evs[es].ebase;
        // an entry pushed while the private stack is full goes to the CTA's shared stack instead
        auto push = [&](const K3Item &c) {
            if (ln < K3F_LSTACK) {
                if (lane == 0) st[ln] = c;
                ++ln;
            } else if (lane == 0) {
                f_lock(S);
                f_place(&S, es, screen, c);
                f_unlock(S);
            }
        };
        if (w < 0) {
            // ---- the window loop of _recursive_split up to the next scannable window (cparsers.pyx:186-193);
            //      every lane runs it, lane 0 writes ----
            bool scan = false;
            for (;;) {
                const long long lim = (long long)it.e - 2LL * mw;
                if (it.ps >= lim) {
                    if (it.e - it.s > MW) {
                        const int x = k3_forced(P, it.s, it.e);
                        if (lane == 0) k3_emit(G, off, x);
                        K3Item l, r;
                        l.s = it.s; l.e = x; l.ps = it.s; l.pad = 0;
                        r.s = x; r.e = it.e; r.ps = x; r.pad = 0;
                        const bool wl = k3_worth(P, l.s, l.e), wr = k3_worth(P, r.s, r.e);
                        if (wl && wr) { push(r); it = l; continue; }
                        if (wl) { it = l; continue; }
                        if (wr) { it = r; continue; }
                    }
                    break;
                }
                if (it.ps > (long long)it.s + MW) {
                    const int x = k3_forced(P, it.s, it.e);
                    if (lane == 0) k3_emit(G, off, x);  // the left part is not revisited (cparsers.pyx:189-191)
                    if (!k3_worth(P, x, it.e)) break;
                    it.s = x; it.ps = x;
                    continue;
                }
                const int pe_t = k3_window_end(P, it);
                if (pe_t - it.ps <= 2 * mw) { it.ps = k3_next_ps(P, it.ps, it.e); continue; }
                scan = true;
                break;
            }
            __syncwarp();
            if (!scan) continue;
        }
        exact = !(screen && ebase != K3_NO_EBASE);

        // ---- scan: one piece of a shared window, or a whole private window --------------------------------
        const double2 *ccg = G.cc + off;
        K3GlobalCC acc;
        acc.g = ccg;
        const int pe = k3_window_end(P, it);
        const int ncand = pe - it.ps - 2 * mw + 1;
        const int nch = (ncand + 31) >> 5;
        if (w < 0) pc = nch;
        const double2 lo = acc.at(it.ps - 1), hi = acc.at(pe - 1);
        unsigned long long K1, K2 = K3_NOKEY;
        int I1;
        {
            const int w_last = pe - mw;
            int i_end = it.ps + mw + (p + 1) * pc * 32 - 1;
            i_end = i_end < w_last ? i_end : w_last;
            const int i0 = it.ps + mw + p * pc * 32 + lane;
            if (!exact) {
                K3Scr a;
                k3_scr_init(a);
                k3_screen_lane(ccg, lo, hi, it.ps, pe, ebase, G.RN, i0, i_end, 32, a);
                bool bad;
                k3_warp_summary(a, K1, K2, I1, bad);
                I1 = ((I1 - it.ps) & 0x1fffffff) | (bad ? K3_BAD_FLAG : 0);
            } else {
                const K3Best b = f_exact_range(ccg, it.ps, pe, i0, i_end, P.min_gain);
                K1 = (unsigned long long)__double_as_longlong(b.g);
                I1 = b.x;
            }
        }
        if (np > 1) {
            K3FWin &Wn = S.win[w];
            int old = 0;
            if (lane == 0) {
                Wn.k1[p] = K1; Wn.k2[p] = K2; Wn.i1[p] = I1;
                __threadfence_block();
                old = atomicAdd(&Wn.done, 1);
                __threadfence_block();
            }
            old = __shfl_sync(PP_FULL, old, 0);
            if (old != np - 1) continue;   // other pieces of the window are still being scanned
            const volatile K3FWin &V = Wn;  // this warp decides: lane q takes piece q's summary
            K1 = lane < np ? V.k1[lane] : K3_NOKEY;
            K2 = lane < np ? V.k2[lane] : K3_NOKEY;
            I1 = lane < np ? V.i1[lane] : -1;
        } else if (lane != 0 && !exact) {   // one piece: its summary sits in lane 0, like piece 0 of a shared window
            K1 = K2 = K3_NOKEY;
            I1 = -1;
        }

        // ---- the window is complete: decide --------------------------------------------------------------
        int x;
        unsigned nexact = 0;
        if (!exact) {
            x = f_decide(G, P, ccg, lo, hi, it.ps, pe, ebase, np, pc, K1, K2, I1, nexact, T.br);
        } else {
            K3Best b;
            b.g = __longlong_as_double((long long)K1);
            b.x = I1;
            if (np > 1) {
                if (lane >= np) { b.g = P.min_gain; b.x = -1; }
                b = k3_warp_reduce(b);
            }
            x = __shfl_sync(PP_FULL, b.x, 0);
            if (screen) {
                nexact = (unsigned)ncand;
                ++T.br.full;
            }
        }
        T.cand += (unsigned long long)ncand;
        T.scans += 1;
        T.exact += nexact;

        // ---- the recursion's bookkeeping (cparsers.pyx:194-203): children small enough stay with this warp, the
        //      others go onto the shared stack; the right child first, so that the left one is resolved first ----
        K3Item big[2];
        int nbig = 0;
        const int ln_before = ln;
        auto child = [&](const K3Item &c) {
            if (w < 0 || c.e - c.s <= K3F_LOCAL) push(c);
            else big[nbig++] = c;
        };
        if (x >= 0) {
            if (lane == 0) k3_emit(G, off, x);
            K3Item c;
            c.pad = 0;
            if (k3_worth(P, x, it.e)) {
                bool away = false;
                if (K3_IDLE_SHARE > 0 && S.few && x - it.s >= K3_IDLE_SHARE && it.e - x >= K3_IDLE_SHARE) {
                    // CTAs waiting for work hold tickets past the queue's tail: hand them the right child
                    // (lane 0 looks, so that every lane takes the same branch)
                    int waiting = 0;
                    if (lane == 0) {
                        const unsigned long long qh = *((volatile unsigned long long *)&G.ctr->q_head);
                        const unsigned long long qt = *((volatile unsigned long long *)&G.ctr->q_tail);
                        waiting = (long long)(qh - qt) > 0 ? 1 : 0;
                    }
                    away = __shfl_sync(PP_FULL, waiting, 0) != 0;
                }
                if (away) {
                    if (lane == 0) f_push_global(G, S.evs[es].ev, x, it.e, x);
                } else {
                    c.s = x; c.e = it.e; c.ps = x;
                    child(c);
                }
            }
            if (k3_worth(P, it.s, x)) { c.s = it.s; c.e = x; c.ps = it.s; child(c); }
        } else {
            it.ps = k3_next_ps(P, it.ps, it.e);
            child(it);
        }
        if (w >= 0) {
            const int keeps = ln > ln_before ? 1 : 0;
            if (lane == 0) f_retire(&S, es, screen, w, big, nbig, keeps);
            if (keeps) les = es;
        }
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(&S.cand, T.cand);
        atomicAdd(&S.scans, T.scans);
        atomicAdd(&S.exact, T.exact);
        if (T.br.sure) atomicAdd(&S.sure, (unsigned long long)T.br.sure);
        if (T.br.multi) atomicAdd(&S.multi, (unsigned long long)T.br.multi);
        if (T.br.full) atomicAdd(&S.full, (unsigned long long)T.br.full);
    }
    __syncthreads();
    if (tid == 0) {
        atomicAdd(&G.ctr->n_cand, S.cand);
        atomicAdd(&G.ctr->n_scan, S.scans);
        atomicAdd(&G.ctr->n_exact, S.exact);
        atomicAdd(&G.ctr->n_tasks, S.tasks);
        if (S.sure) atomicAdd(&G.ctr->n_sure, S.sure);
        if (S.multi) atomicAdd(&G.ctr->n_multi, S.multi);
        if (S.full) atomicAdd(&G.ctr->n_full, S.full);
    }
}
