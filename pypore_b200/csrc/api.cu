// api.cu -- C ABI of libpypore_b200.so (see include/pypore_b200.h).
//
// Host-side plumbing only: buffer management, stream-ordered kernel launches,
// counters read-back.  All arithmetic lives in the kernels.
#include "common.cuh"
#include "threshold.cuh"
#include "prefix.cuh"
#include "split.cuh"
#include "split_flow.cuh"
#include "stats.cuh"
#include "filter.cuh"
#include "hmm.cuh"

#include <new>
#include <stdarg.h>
#include <stdlib.h>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only (no link dependency); ranges cost nothing without a profiler attached

namespace {

// Device memory that belongs to one owner (a pp_ctx member or a scratch local) and is freed with it
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;

    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            if (p) cudaFree(p);
            p = std::exchange(o.p, nullptr);
            cap = std::exchange(o.cap, 0);
        }
        return *this;
    }
    ~DevBuf() { if (p) cudaFree(p); }
};

enum { ST_THRESHOLD = 0, ST_SELECT, ST_FILTER, ST_PREFIX, ST_SPLIT, ST_COMPACT, ST_STATS, ST_COUNT };

// NVTX range over the host-side enqueue of a stage (SURVEY section 5: tracing); shows up in Nsight Systems next to
// the kernels it launched
struct StageRange {
    explicit StageRange(const char *name) { nvtxRangePushA(name); }
    ~StageRange() { nvtxRangePop(); }
};

}  // namespace

struct pp_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    char err[512] = {0};
    int64_t launches = 0;

    // trace: the resident samples (in trace_buf, or adopted), float32, float64 or int16 ADC counts (decoded with adc)
    // as trace_kind (PP_SRC_*) says
    DevBuf trace_buf;
    const void *trace = nullptr;
    int trace_kind = PP_SRC_TRACE32;
    // pp_trace_prefetch: up to two float32 traces on their way up while the resident one is processed (oldest first);
    // trace_spare is the buffer the last swap retired
    struct Pending {
        DevBuf buf;
        int64_t n = -1;
        cudaEvent_t done = nullptr, t0 = nullptr, t1 = nullptr;
    } pend[2];
    int n_pend = 0;
    DevBuf trace_spare;
    PPAdc adc = {1.0, 0.0};
    int64_t n = 0, trace_cap = 0;

    // counters
    PPCounters *ctr = nullptr;
    PPCounters *h_ctr = nullptr;  // pinned

    // K1
    DevBuf k1_rec, k1_staged, k1_blk, run_start, run_minkey, run_maxkey, run_len, run_min, run_max, run_below;
    int64_t cap_runs = 0;
    int64_t n_runs = -1;
    int64_t scan_len = 0;
    int64_t k1_tiles_done = 0;  // tiles scanned so far (the streamed pipeline scans chunk after chunk)
    int k1_flip = 0;            // which n_edges slot the next k1_stitch reads

    // events
    DevBuf ev_start, ev_len, ev_off;
    int64_t cap_events = 0;
    int64_t n_events = -1, n_event_samples = -1;
    int src_kind = 0;
    DevBuf flat64;       // kind 1 samples / filtered current
    int64_t flat_cap = 0;  // capacity in samples of flat event space for the current source

    // K2/K3
    DevBuf cc, bits, tasks, ready, block_count, block_off, inexact, Ttab, ev_tile_off, k2_bits, k2_tiles;
    DevBuf hk;  // K3_CFG_HALFKEY development variant: half-keys, 2 x 8 B per flat sample
    DevBuf unpack_flag;
    // multi-GPU control exchange over peer memory (pp_ctl_*)
    DevBuf ctl_buf, ctl_peers_dev;
    void *ctl_peers[64] = {nullptr};
    bool ctl_ipc[64] = {false};
    int ctl_rank = -1, ctl_world = 0;
    unsigned long long ctl_seq = 0;
    int opt_spine = 1;
    int T_len = 0;
    int opt_screen = 1;
    int opt_split_ctas = 0;  // 0: one full wave (K3_CTAS_PER_SM per SM)
    int opt_split_kernel = PP_SPLIT_KERNEL_DEFAULT;  // 0: k3_split (level-synchronous CTAs), 1: k3_flow (barrier-free warps)
    int64_t q_cap = 0;
    DevBuf seg_flat, seg_event, seg_start, seg_end, seg_mean, seg_std, seg_min, seg_max;
    int64_t cap_segs = 0;
    int64_t n_segments = -1;
    bool stats_valid = false;
    int64_t split_counters[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    bool prefix_valid = false;  // cc holds the prefix sums of the current events
    int prefix_mode = PP_PREFIX_AUTO;  // mode of the last K2 run (what `inexact` means for pp_debug_prefix)

    // event stats
    DevBuf evs_mean, evs_std, evs_min, evs_max;

    // filter scratch
    DevBuf filt_tmp, filt_carry, filt_coef;

    // HMM decoding (pp_hmm_*): model block, host sequences and their offsets, results of the last decode
    DevBuf hmm_model, hmm_x, hmm_off, hmm_logp, hmm_state, hmm_bp, hmm_next, hmm_old_flat, hmm_old_state;
    int64_t hmm_n_seq = -1, hmm_n_rows = -1;
    bool hmm_states = false;   // the last decode was a Viterbi decode

    // streamed pipeline (pp_pipeline_host): copies run on their own stream
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copy_ev = nullptr, compute_ev = nullptr;
    cudaEvent_t pf_t0 = nullptr, pf_t1 = nullptr;   // timing of the last pp_trace_prefetch copy
    int64_t n_words = 0, n_blocks = 0;

    cudaEvent_t ev[ST_COUNT + 1] = {0};
    bool stage_ran[ST_COUNT] = {false};
    bool rec[ST_COUNT + 1] = {false};  // boundary i recorded in the current call sequence
};

namespace {

int fail(pp_ctx *c, int code, const char *fmt, ...)
{
    if (c) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(c->err, sizeof c->err, fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(ctx, PP_ERR_CUDA, "%s failed: %s (%s:%d)", #call,                 \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                      \
    } while (0)

#define CKR(call)                              \
    do {                                       \
        int r_ = (call);                       \
        if (r_ != PP_OK) return r_;            \
    } while (0)

#define LAUNCHED(ctx)                                                                     \
    do {                                                                                  \
        (ctx)->launches++;                                                                \
        cudaError_t e_ = cudaGetLastError();                                              \
        if (e_ != cudaSuccess)                                                            \
            return fail(ctx, PP_ERR_CUDA, "kernel launch failed: %s (%s:%d)",             \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                      \
    } while (0)

int ensure(pp_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap && b.p) return PP_OK;
    bytes = (bytes + 255) & ~(size_t)255;   // whole 256-byte units: vector loads may touch the rest of a row's last 16 bytes
    CK(cudaStreamSynchronize(ctx->stream));
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    CK(cudaMalloc(&b.p, bytes));
    b.cap = bytes;
    return PP_OK;
}

// Host scratch freed with its scope; a failed allocation is reported, not thrown across the C ABI
template <typename T>
int host_scratch(pp_ctx *ctx, std::vector<T> &v, size_t n)
{
    try {
        v.resize(n);
    } catch (const std::exception &) {
        return fail(ctx, PP_ERR_ARG, "out of host memory");
    }
    return PP_OK;
}

int set_device(pp_ctx *ctx)
{
    CK(cudaSetDevice(ctx->device));
    return PP_OK;
}

int record_boundary(pp_ctx *ctx, int i)
{
    CK(cudaEventRecord(ctx->ev[i], ctx->stream));
    ctx->rec[i] = true;
    return PP_OK;
}

void reset_stages(pp_ctx *ctx)
{
    for (int i = 0; i < ST_COUNT; ++i) ctx->stage_ran[i] = false;
    for (int i = 0; i <= ST_COUNT; ++i) ctx->rec[i] = false;
}

// A call whose stages pp_stage_ms times: earlier boundaries are forgotten, the first one is recorded now
int begin_call(pp_ctx *ctx, int first_boundary)
{
    CKR(set_device(ctx));
    reset_stages(ctx);
    return record_boundary(ctx, first_boundary);
}

// stage `st` is enqueued: the boundary that ends it
int end_stage(pp_ctx *ctx, int st)
{
    CKR(record_boundary(ctx, st + 1));
    ctx->stage_ran[st] = true;
    return PP_OK;
}

// State derived from the trace, each level from the one before it: dropping a level drops the levels after it too
enum { LV_RUNS, LV_EVENTS, LV_PREFIX, LV_SEGMENTS, LV_STATS };

void drop_from(pp_ctx *ctx, int level)
{
    if (level <= LV_RUNS) ctx->n_runs = -1;
    if (level <= LV_EVENTS) ctx->n_events = ctx->n_event_samples = -1;
    if (level <= LV_PREFIX) ctx->prefix_valid = false;
    if (level <= LV_SEGMENTS) ctx->n_segments = -1;
    ctx->stats_valid = false;
}

size_t sample_bytes(int kind)
{
    return kind == PP_SRC_TRACE64 ? sizeof(double) : kind == PP_SRC_ADC16 ? sizeof(int16_t) : sizeof(float);
}

// `n` samples of `kind` at `p` (room for `cap`) become the resident trace
void set_trace(pp_ctx *ctx, const void *p, int kind, int64_t n, int64_t cap)
{
    ctx->trace = p;
    ctx->trace_kind = kind;
    ctx->n = n;
    ctx->trace_cap = cap;
    drop_from(ctx, LV_RUNS);
}

// the resident samples as T if they are of `kind`, else null
template <typename T>
const T *trace_as(const pp_ctx *ctx, int kind)
{
    return ctx->trace_kind == kind ? (const T *)ctx->trace : nullptr;
}

// Which resident traces a call takes: bits 1 << PP_SRC_* of the trace kinds, TAKES_NONE for no trace at all
enum : unsigned {
    TAKES_F32 = 1u << PP_SRC_TRACE32,
    TAKES_NONE = 1u << 8,
    NOT_ADC = TAKES_F32 | 1u << PP_SRC_TRACE64 | TAKES_NONE,
};

int require_trace(pp_ctx *ctx, unsigned takes, const char *what)
{
    if (takes & (ctx->trace ? 1u << ctx->trace_kind : TAKES_NONE)) return PP_OK;
    const char *have = !ctx->trace ? "no trace" : ctx->trace_kind == PP_SRC_ADC16 ? "an ADC trace"
                       : ctx->trace_kind == PP_SRC_TRACE64 ? "a float64 trace" : "a float32 trace";
    return fail(ctx, PP_ERR_STATE, "%s; %s is resident", what, have);
}

PPSource make_source(pp_ctx *ctx)
{
    PPSource s;
    s.trace = trace_as<float>(ctx, PP_SRC_TRACE32);
    s.trace64 = trace_as<double>(ctx, PP_SRC_TRACE64);
    s.trace16 = trace_as<int16_t>(ctx, PP_SRC_ADC16);
    s.adc = ctx->adc;
    s.flat = (const double *)ctx->flat64.p;
    s.ev_start = (const int64_t *)ctx->ev_start.p;
    s.ev_off = (const int64_t *)ctx->ev_off.p;
    s.kind = ctx->src_kind;
    return s;
}

// float64 samples of the current events and the table that locates an event in them
const double *f64_samples(pp_ctx *ctx)
{
    return ctx->src_kind == PP_SRC_TRACE64 ? (const double *)ctx->trace : (const double *)ctx->flat64.p;
}
const int64_t *f64_bases(pp_ctx *ctx)
{
    return (const int64_t *)(ctx->src_kind == PP_SRC_TRACE64 ? ctx->ev_start.p : ctx->ev_off.p);
}

int fetch_counters(pp_ctx *ctx)
{
    CK(cudaMemcpyAsync(ctx->h_ctr, ctx->ctr, sizeof(PPCounters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int ensure_run_buffers(pp_ctx *ctx, int64_t cap_runs)
{
    if (cap_runs <= ctx->cap_runs) return PP_OK;
    CKR(ensure(ctx, ctx->run_start, sizeof(int64_t) * cap_runs));
    CKR(ensure(ctx, ctx->run_minkey, sizeof(unsigned long long) * cap_runs));
    CKR(ensure(ctx, ctx->run_maxkey, sizeof(unsigned long long) * cap_runs));
    CKR(ensure(ctx, ctx->run_len, sizeof(int64_t) * cap_runs));
    CKR(ensure(ctx, ctx->run_min, sizeof(double) * cap_runs));
    CKR(ensure(ctx, ctx->run_max, sizeof(double) * cap_runs));
    CKR(ensure(ctx, ctx->run_below, cap_runs));
    ctx->cap_runs = cap_runs;
    return PP_OK;
}

int ensure_event_buffers(pp_ctx *ctx, int64_t cap_events)
{
    if (cap_events <= ctx->cap_events) return PP_OK;
    CKR(ensure(ctx, ctx->ev_start, sizeof(int64_t) * (cap_events + 1)));
    CKR(ensure(ctx, ctx->ev_len, sizeof(int64_t) * (cap_events + 1)));
    CKR(ensure(ctx, ctx->ev_off, sizeof(int64_t) * (cap_events + 1)));
    ctx->cap_events = cap_events;
    return PP_OK;
}

// ---- stage enqueue helpers (no host synchronisation) ----------------------

// Buffers and zeroed state for a threshold scan of the first scan_len samples.
int begin_threshold(pp_ctx *ctx, int64_t scan_len)
{
    ctx->scan_len = scan_len;
    // one run per 256 samples to begin with (the headline traces have one per 6000); a noisier trace overflows once,
    // the table is regrown to what the scan counted and the call repeats (the capacity stays with the context)
    int64_t want = scan_len / 256 + 4096;
    if (want < ctx->cap_runs) want = ctx->cap_runs;
    CKR(ensure_run_buffers(ctx, want));
    CKR(ensure_event_buffers(ctx, ctx->cap_runs));
    const int64_t ntiles = (scan_len + K1_TILE - 1) / K1_TILE;
    const int64_t nrec = ntiles * K1_WARPS;
    CKR(ensure(ctx, ctx->k1_rec, sizeof(K1Record) * nrec));
    CKR(ensure(ctx, ctx->k1_staged, sizeof(K1Staged) * nrec * K1_STAGE));
    CKR(ensure(ctx, ctx->k1_blk, sizeof(unsigned long long) * ((nrec + K1B_THREADS - 1) / K1B_THREADS + 1)));
    CK(cudaMemsetAsync(ctx->ctr, 0, sizeof(PPCounters), ctx->stream));
    CK(cudaMemsetAsync(ctx->run_minkey.p, 0xff, sizeof(unsigned long long) * ctx->cap_runs, ctx->stream));
    CK(cudaMemsetAsync(ctx->run_maxkey.p, 0, sizeof(unsigned long long) * ctx->cap_runs, ctx->stream));
    ctx->k1_tiles_done = 0;
    ctx->k1_flip = 0;
    drop_from(ctx, LV_RUNS);
    return PP_OK;
}

template <typename T>
int launch_threshold_tiles(pp_ctx *ctx, const T *x, typename K1Key<T>::V thr, int kxor, int64_t upto,
                           int64_t tile_begin, int64_t ntiles)
{
    const size_t smem = sizeof(K1Smem<T>);
    static int per_sm = 0;   // per instantiation: resident CTAs per SM (the kernel is persistent: one wave exactly)
    if (per_sm == 0) {
        CK(cudaFuncSetAttribute(k1_scan_tiles<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k1_scan_tiles<T>, K1_CTA_THREADS, smem));
        per_sm = nb > 0 ? nb : 1;
    }
    int64_t grid = (int64_t)ctx->sm_count * per_sm;
    if (grid > ntiles) grid = ntiles;
    k1_scan_tiles<T><<<(unsigned)grid, K1_CTA_THREADS, smem, ctx->stream>>>(
        x, upto, thr, kxor, tile_begin, ntiles, (K1Record *)ctx->k1_rec.p, (K1Staged *)ctx->k1_staged.p);
    LAUNCHED(ctx);
    const int64_t rec_begin = tile_begin * K1_WARPS, rec_end = (tile_begin + ntiles) * K1_WARPS;
    const int64_t nblk = (rec_end - rec_begin + K1B_THREADS - 1) / K1B_THREADS;
    CK(cudaMemsetAsync(ctx->k1_blk.p, 0, sizeof(unsigned long long) * nblk, ctx->stream));
    k1_stitch<T><<<(unsigned)nblk, K1B_THREADS, 0, ctx->stream>>>(
        x, upto, thr, kxor, rec_begin, rec_end, (const K1Record *)ctx->k1_rec.p, (const K1Staged *)ctx->k1_staged.p,
        (unsigned long long *)ctx->k1_blk.p, ctx->ctr, ctx->k1_flip, (int64_t *)ctx->run_start.p,
        (unsigned long long *)ctx->run_minkey.p, (unsigned long long *)ctx->run_maxkey.p, ctx->cap_runs);
    LAUNCHED(ctx);
    ctx->k1_flip ^= 1;
    return PP_OK;
}

// Scan the next `ntiles` tiles (the tile counter continues across calls) of the trace prefix
// [0, upto) and decode the run table found so far.
int enqueue_threshold_tiles(pp_ctx *ctx, double threshold, int64_t upto, int64_t ntiles)
{
    StageRange nvtx_range("pypore:threshold");
    if (ntiles > 0) {
        if (ctx->trace_kind == PP_SRC_TRACE64) {
            CKR(launch_threshold_tiles<double>(ctx, (const double *)ctx->trace, threshold, 0, upto, ctx->k1_tiles_done,
                                               ntiles));
        } else if (ctx->trace_kind == PP_SRC_ADC16) {
            int32_t key = 0, kxor = 0;
            pp_adc16_key_threshold(ctx->adc.scale, ctx->adc.offset, threshold, &key, &kxor);
            CKR(launch_threshold_tiles<int16_t>(ctx, (const int16_t *)ctx->trace, key, kxor, upto, ctx->k1_tiles_done,
                                                ntiles));
        } else {
            // smallest float32 >= threshold: double(x) < thr  <=>  x < thr_up for every float32 x
            float thr_f = (float)threshold;
            if ((double)thr_f < threshold) thr_f = nextafterf(thr_f, INFINITY);
            CKR(launch_threshold_tiles<float>(ctx, (const float *)ctx->trace, thr_f, 0, upto, ctx->k1_tiles_done,
                                              ntiles));
        }
        ctx->k1_tiles_done += ntiles;
    }
    k1_finalize_runs<<<ctx->sm_count, 256, 0, ctx->stream>>>(
        upto, ctx->ctr, (const int64_t *)ctx->run_start.p, (const unsigned long long *)ctx->run_minkey.p,
        (const unsigned long long *)ctx->run_maxkey.p, ctx->cap_runs, (int64_t *)ctx->run_len.p,
        (double *)ctx->run_min.p, (double *)ctx->run_max.p, (unsigned char *)ctx->run_below.p,
        ctx->trace_kind == PP_SRC_ADC16, ctx->adc);
    LAUNCHED(ctx);
    return PP_OK;
}

int enqueue_threshold(pp_ctx *ctx, double threshold, int64_t scan_len)
{
    if (!ctx->trace || ctx->n <= 0) return fail(ctx, PP_ERR_STATE, "no trace resident");
    if (scan_len < 0 || scan_len > ctx->n) scan_len = ctx->n;
    CKR(begin_threshold(ctx, scan_len));
    return enqueue_threshold_tiles(ctx, threshold, scan_len, (scan_len + K1_TILE - 1) / K1_TILE);
}

int enqueue_select(pp_ctx *ctx, int rule_mask, int64_t duration_gt, int64_t duration_lt,
                   double min_gt, double max_lt, int skip_first, int skip_last, int incremental = 0,
                   const long long *dev_plan = nullptr)
{
    StageRange nvtx_range("pypore:select");
    ctx->src_kind = ctx->trace_kind;
    ctx->flat_cap = ctx->n;
    k1_select_events<<<1, SEL_THREADS, 0, ctx->stream>>>(
        ctx->ctr, (const int64_t *)ctx->run_start.p, (const int64_t *)ctx->run_len.p,
        (const double *)ctx->run_min.p, (const double *)ctx->run_max.p, ctx->cap_runs, rule_mask,
        duration_gt, duration_lt, min_gt, max_lt, skip_first, skip_last, (int64_t *)ctx->ev_start.p,
        (int64_t *)ctx->ev_len.p, (int64_t *)ctx->ev_off.p, ctx->cap_events, incremental, dev_plan);
    LAUNCHED(ctx);
    drop_from(ctx, LV_EVENTS);
    return PP_OK;
}

template <int NZ>
void launch_filter_sequential(pp_ctx *ctx, const PPSource &src, int backward)
{
    k5_filter_sequential<NZ><<<ctx->sm_count * 8, 64, 0, ctx->stream>>>(
        src, (const int64_t *)ctx->ev_len.p, ctx->ctr, (const K5Coef *)ctx->filt_coef.p,
        (double *)ctx->filt_tmp.p, (double *)ctx->flat64.p, backward);
}

template <int NZ>
void launch_filter_pass(pp_ctx *ctx, const PPSource &src, int backward)
{
    cudaFuncSetAttribute(k5_filter_pass<NZ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)k5_smem_bytes<NZ>());
    k5_filter_pass<NZ><<<ctx->sm_count * 4, K5_THREADS, k5_smem_bytes<NZ>(), ctx->stream>>>(
        src, (const int64_t *)ctx->ev_len.p, ctx->ctr, (const K5Coef *)ctx->filt_coef.p,
        (double *)ctx->filt_tmp.p, (double *)ctx->flat64.p, backward);
}

int enqueue_filter(pp_ctx *ctx, const double *b, const double *a, const double *zi, int nc)
{
    StageRange nvtx_range("pypore:filter");
    if (nc < 2 || nc > FILT_MAX_COEF) return fail(ctx, PP_ERR_ARG, "filter order must be 1..%d", FILT_NZ);
    if (a[0] != 1.0) return fail(ctx, PP_ERR_ARG, "filter coefficients must be normalised (a[0] == 1)");
    const int64_t ncap = ctx->flat_cap;
    if (ncap <= 0) return fail(ctx, PP_ERR_STATE, "no events selected");
    const int P = 3 * nc;
    int64_t max_events = ncap / (P + 1) + 1;
    if (ctx->n_events >= 0 && ctx->n_events < max_events) max_events = ctx->n_events;
    if (ctx->cap_events < max_events) max_events = ctx->cap_events;
    CKR(ensure(ctx, ctx->filt_tmp, sizeof(double) * (size_t)(ncap + 2 * P * max_events + 64)));
    CKR(ensure(ctx, ctx->flat64, sizeof(double) * (size_t)ncap));
    CKR(ensure(ctx, ctx->filt_coef, sizeof(K5Coef)));
    K5Coef C;
    k5_prepare(b, a, zi, nc, &C);
    CK(cudaMemcpyAsync(ctx->filt_coef.p, &C, sizeof C, cudaMemcpyHostToDevice, ctx->stream));
    for (int backward = 0; backward < 2; ++backward) {
        PPSource src = make_source(ctx);
        switch (nc - 1) {
        case 1: launch_filter_pass<1>(ctx, src, backward); break;
        case 2: launch_filter_pass<2>(ctx, src, backward); break;
        case 3: launch_filter_sequential<3>(ctx, src, backward); break;
        case 4: launch_filter_sequential<4>(ctx, src, backward); break;
        case 5: launch_filter_sequential<5>(ctx, src, backward); break;
        case 6: launch_filter_sequential<6>(ctx, src, backward); break;
        case 7: launch_filter_sequential<7>(ctx, src, backward); break;
        default: launch_filter_sequential<8>(ctx, src, backward); break;
        }
        LAUNCHED(ctx);
    }
    ctx->src_kind = PP_SRC_FLAT64;  // from here on the events' current is the filtered float64 signal
    CKR(end_stage(ctx, ST_FILTER));
    drop_from(ctx, LV_PREFIX);
    return PP_OK;
}

// Argument checks and buffers for K2/K3/compaction, sized by upper bounds (no host sync later).
int prepare_split(pp_ctx *ctx, int mw, int MW, int W)
{
    if (mw < 0 || MW < mw || W < 2 * mw || W / 2 < 1)
        return fail(ctx, PP_ERR_ARG, "invalid split parameters (min_width=%d max_width=%d window_width=%d)",
                    mw, MW, W);
    const int64_t ncap = ctx->flat_cap;
    if (ncap <= 0) return fail(ctx, PP_ERR_STATE, "no events selected");
    // a forced max_width split min(s + MW, e - mw) may leave ONE piece shorter than min_width next to one that is at
    // least min_width long (mw = MW = 100: 150 samples -> 50 + 100), so segments average at least min_width / 2
    const int64_t div = mw > 0 ? mw : 1;
    const int64_t cap_segs = 2 * (ncap / div) + ctx->cap_events + 16;
    const int64_t q_cap = ctx->cap_events + 2 * (ncap / div) + 1024;
    const int64_t n_words = (ncap + 31) / 32 + 1;
    const int64_t n_blocks = (n_words + CP_BLOCK_WORDS - 1) / CP_BLOCK_WORDS;
    CKR(ensure(ctx, ctx->cc, sizeof(double2) * ncap));
    CKR(ensure(ctx, ctx->bits, sizeof(unsigned) * n_words));
    CKR(ensure(ctx, ctx->tasks, sizeof(PPTask) * q_cap));
    CKR(ensure(ctx, ctx->ready, sizeof(int) * q_cap));
    CKR(ensure(ctx, ctx->block_count, sizeof(unsigned) * n_blocks));
    CKR(ensure(ctx, ctx->block_off, sizeof(unsigned long long) * n_blocks));
    if (cap_segs > ctx->cap_segs) {
        CKR(ensure(ctx, ctx->seg_flat, sizeof(int64_t) * cap_segs));
        CKR(ensure(ctx, ctx->seg_event, sizeof(int) * cap_segs));
        CKR(ensure(ctx, ctx->seg_start, sizeof(int64_t) * cap_segs));
        CKR(ensure(ctx, ctx->seg_end, sizeof(int64_t) * cap_segs));
        CKR(ensure(ctx, ctx->seg_mean, sizeof(double) * cap_segs));
        CKR(ensure(ctx, ctx->seg_std, sizeof(double) * cap_segs));
        CKR(ensure(ctx, ctx->seg_min, sizeof(double) * cap_segs));
        CKR(ensure(ctx, ctx->seg_max, sizeof(double) * cap_segs));
        ctx->cap_segs = cap_segs;
    }
    ctx->q_cap = q_cap;
    ctx->n_words = n_words;
    ctx->n_blocks = n_blocks;
    if (W + 1 > ctx->T_len) {
        CKR(ensure(ctx, ctx->Ttab, sizeof(double) * (size_t)(W + 1)));
        k3_fill_RN<<<ctx->sm_count, 256, 0, ctx->stream>>>((double *)ctx->Ttab.p, W + 1);
        LAUNCHED(ctx);
        ctx->T_len = W + 1;
    }
    CK(cudaMemsetAsync(ctx->bits.p, 0, sizeof(unsigned) * n_words, ctx->stream));
    CK(cudaMemsetAsync(&ctx->ctr->seg_done, 0, 3 * sizeof(unsigned long long), ctx->stream));  // seg/flat/ev_done
    return PP_OK;
}

// K2's tiled scan with the exactness proof over the samples `samples` of the event source `src`
template <typename T>
int enqueue_prefix_tiled(pp_ctx *ctx, const PPSource &src, const T *samples, int prefix_mode)
{
    // short events: one pass, one warp per event
    k2_event_scan<T><<<ctx->sm_count * K2F_CFG_CTAS * 2, K2F_WARPS * 32, 0, ctx->stream>>>(
        src, samples, (const int64_t *)ctx->ev_len.p, ctx->ctr, (unsigned *)ctx->inexact.p, (double2 *)ctx->cc.p,
        prefix_mode != PP_PREFIX_PARALLEL);
    LAUNCHED(ctx);
    // long events: multi-CTA reduce / carries / scan over their tiles
    const int grid = ctx->sm_count * 8;
    k2_tile_reduce<T><<<grid, K2_THREADS, 0, ctx->stream>>>(
        src, samples, (const int64_t *)ctx->ev_len.p, (const int64_t *)ctx->ev_tile_off.p, ctx->ctr,
        (K2TileState *)ctx->k2_tiles.p, (K2EventBits *)ctx->k2_bits.p);
    LAUNCHED(ctx);
    k2_event_carries<<<ctx->sm_count * 2, 256, 0, ctx->stream>>>(
        ctx->ctr, (const int64_t *)ctx->ev_len.p, (const int64_t *)ctx->ev_tile_off.p,
        (K2TileState *)ctx->k2_tiles.p, (const K2EventBits *)ctx->k2_bits.p, (unsigned *)ctx->inexact.p,
        prefix_mode != PP_PREFIX_PARALLEL);
    LAUNCHED(ctx);
    k2_tile_scan<T><<<grid, K2_THREADS, 0, ctx->stream>>>(
        src, samples, (const int64_t *)ctx->ev_len.p, (const int64_t *)ctx->ev_tile_off.p, ctx->ctr,
        (const K2TileState *)ctx->k2_tiles.p, (double2 *)ctx->cc.p);
    LAUNCHED(ctx);
    return PP_OK;
}

// K2 over the events [ev_begin, n_events) (device-side range)
int enqueue_prefix(pp_ctx *ctx, int prefix_mode)
{
    StageRange nvtx_range("pypore:prefix");
    const int64_t ncap = ctx->flat_cap;
    PPSource src = make_source(ctx);
    ctx->prefix_mode = prefix_mode;
    if (prefix_mode == PP_PREFIX_SEQUENTIAL) {
        k2_prefix_sequential<<<ctx->sm_count * 3, K2S_WARPS * 32, 0, ctx->stream>>>(
            src, (const int64_t *)ctx->ev_len.p, ctx->ctr, nullptr, (double2 *)ctx->cc.p);
        LAUNCHED(ctx);
    } else {
        const int64_t max_tiles = ncap / K2_TILE + ctx->cap_events + 2;
        CKR(ensure(ctx, ctx->ev_tile_off, sizeof(int64_t) * (ctx->cap_events + 2)));
        CKR(ensure(ctx, ctx->k2_bits, sizeof(K2EventBits) * (ctx->cap_events + 1)));
        CKR(ensure(ctx, ctx->inexact, sizeof(unsigned) * (ctx->cap_events + 1)));
        CKR(ensure(ctx, ctx->k2_tiles, sizeof(K2TileState) * (size_t)max_tiles));
        k2_tile_offsets<<<1, 1024, 0, ctx->stream>>>(ctx->ctr, (const int64_t *)ctx->ev_len.p,
                                                     (int64_t *)ctx->ev_tile_off.p, (K2EventBits *)ctx->k2_bits.p,
                                                     (unsigned *)ctx->inexact.p);
        LAUNCHED(ctx);
        if (ctx->src_kind == PP_SRC_TRACE32) CKR(enqueue_prefix_tiled<float>(ctx, src, src.trace, prefix_mode));
        else if (ctx->src_kind == PP_SRC_ADC16) CKR(enqueue_prefix_tiled<int16_t>(ctx, src, src.trace16, prefix_mode));
        else CKR(enqueue_prefix_tiled<double>(ctx, src, f64_samples(ctx), prefix_mode));
        if (prefix_mode != PP_PREFIX_PARALLEL) {
            k2_prefix_sequential<<<ctx->sm_count * 3, K2S_WARPS * 32, 0, ctx->stream>>>(
                src, (const int64_t *)ctx->ev_len.p, ctx->ctr, (const unsigned *)ctx->inexact.p,
                (double2 *)ctx->cc.p);
            LAUNCHED(ctx);
        }
    }
    return PP_OK;
}

// K3 over the events [ev_begin, n_events)
int enqueue_search(pp_ctx *ctx, int mw, int MW, int W, double min_gain)
{
    StageRange nvtx_range("pypore:split");
    const int64_t q_cap = ctx->q_cap;
    CK(cudaMemsetAsync(ctx->ready.p, 0, sizeof(int) * q_cap, ctx->stream));
    K3Global G;
    G.cc = (const double2 *)ctx->cc.p;
    G.ev_off = (const int64_t *)ctx->ev_off.p;
    G.ev_len = (const int64_t *)ctx->ev_len.p;
    G.bits = (unsigned *)ctx->bits.p;
    G.tasks = (PPTask *)ctx->tasks.p;
    G.ready = (int *)ctx->ready.p;
    G.q_cap = q_cap;
    G.ctr = ctx->ctr;
    if (W + 1 > ctx->T_len) {
        CKR(ensure(ctx, ctx->Ttab, sizeof(double) * (size_t)(W + 1)));
        k3_fill_RN<<<ctx->sm_count, 256, 0, ctx->stream>>>((double *)ctx->Ttab.p, W + 1);
        LAUNCHED(ctx);
        ctx->T_len = W + 1;
    }
    G.RN = (const double *)ctx->Ttab.p;
    G.screen = ctx->opt_screen;
#if K3_CFG_HALFKEY
    CKR(ensure(ctx, ctx->hk, 2 * sizeof(unsigned long long) * (size_t)ctx->flat_cap));
    G.hkL = (unsigned long long *)ctx->hk.p;
    G.hkR = G.hkL + ctx->flat_cap;
#endif
    K3Params P;
    P.mw = mw; P.MW = MW; P.W = W; P.min_gain = min_gain;
    k3_init_queue<<<ctx->sm_count, 256, 0, ctx->stream>>>(G, ctx->opt_spine);
    LAUNCHED(ctx);
    if (ctx->opt_spine) {  // events longer than K3_CAP: their window chain first, a whole CTA per scan
        k3_spine<<<(ctx->sm_count / K3S_CLUSTER) * K3S_CLUSTER, K3S_THREADS, 0, ctx->stream>>>(G, P);
        LAUNCHED(ctx);
    }
    // the queue is served by however many CTAs there are; contexts that share the GPU (file batches) take a
    // fraction of a wave each so that their searches are resident side by side
    const int wave = ctx->sm_count * (ctx->opt_split_kernel ? K3F_CTAS_PER_SM : K3_CTAS_PER_SM);
    const int k3_grid = ctx->opt_split_ctas > 0 && ctx->opt_split_ctas < wave ? ctx->opt_split_ctas : wave;
    if (ctx->opt_split_kernel)
        k3_flow<<<k3_grid, K3F_THREADS, K3F_SMEM_BYTES, ctx->stream>>>(G, P);
    else
        k3_split<<<k3_grid, K3_THREADS, K3_SMEM_BYTES, ctx->stream>>>(G, P);
    LAUNCHED(ctx);
    return PP_OK;
}

// bitmap -> segment table over the flat range not finalised yet (all events unless the streamed pipeline exports
// per chunk)
int enqueue_compact(pp_ctx *ctx)
{
    StageRange nvtx_range("pypore:compact");
    const int64_t n_blocks = ctx->n_blocks;
    k3c_count<<<(unsigned)n_blocks, CP_THREADS, 0, ctx->stream>>>((const unsigned *)ctx->bits.p, ctx->ctr,
                                                                 (unsigned *)ctx->block_count.p);
    LAUNCHED(ctx);
    k3c_scan<<<1, 1024, 0, ctx->stream>>>((const unsigned *)ctx->block_count.p,
                                          (unsigned long long *)ctx->block_off.p, ctx->ctr, ctx->cap_segs);
    LAUNCHED(ctx);
    k3c_write<<<(unsigned)n_blocks, CP_THREADS, 0, ctx->stream>>>(
        (const unsigned *)ctx->bits.p, (const unsigned long long *)ctx->block_off.p,
        (const int64_t *)ctx->ev_off.p, ctx->ctr, (int64_t *)ctx->seg_flat.p, (int *)ctx->seg_event.p,
        (int64_t *)ctx->seg_start.p, ctx->cap_segs);
    LAUNCHED(ctx);
    k3c_ends<<<ctx->sm_count, 256, 0, ctx->stream>>>(ctx->ctr, (const int64_t *)ctx->seg_flat.p,
                                                     (const int *)ctx->seg_event.p,
                                                     (const int64_t *)ctx->ev_off.p,
                                                     (int64_t *)ctx->seg_end.p, ctx->cap_segs);
    LAUNCHED(ctx);
    return PP_OK;
}

// rows / events finalised since the last call -> page-locked host tables, then the range advances
int enqueue_export(pp_ctx *ctx, const PPHostTables &H, int with_stats)
{
    StageRange nvtx_range("pypore:export");
    k_export_tables<<<ctx->sm_count * 2, 256, 0, ctx->stream>>>(
        ctx->ctr, H, (const int64_t *)ctx->ev_start.p, (const int64_t *)ctx->ev_len.p, (const int *)ctx->seg_event.p,
        (const int64_t *)ctx->seg_start.p, (const int64_t *)ctx->seg_end.p, (const double *)ctx->seg_mean.p,
        (const double *)ctx->seg_std.p, (const double *)ctx->seg_min.p, (const double *)ctx->seg_max.p, with_stats);
    LAUNCHED(ctx);
    k_tables_advance<<<1, 32, 0, ctx->stream>>>(ctx->ctr);
    LAUNCHED(ctx);
    return PP_OK;
}

int enqueue_split(pp_ctx *ctx, int mw, int MW, int W, double min_gain, int prefix_mode)
{
    CKR(prepare_split(ctx, mw, MW, W));
    CKR(enqueue_prefix(ctx, prefix_mode));
    ctx->prefix_valid = true;
    drop_from(ctx, LV_SEGMENTS);
    CKR(end_stage(ctx, ST_PREFIX));
    CKR(enqueue_search(ctx, mw, MW, W, min_gain));
    CKR(end_stage(ctx, ST_SPLIT));
    CKR(enqueue_compact(ctx));
    return end_stage(ctx, ST_COMPACT);
}

// K4 over the rows of the current event source: segments (flat_start = seg_flat, row_event = seg_event) or whole
// events (rows_are_events, flat_start = ev_off, row_event = nullptr)
int launch_stats(pp_ctx *ctx, int rows_are_events, const int64_t *flat_start, const int *row_event, int64_t cap_rows,
                 double *mean, double *sd, double *mn, double *mx)
{
    const unsigned grid = ctx->sm_count * 8;
    const int64_t *ev_off = (const int64_t *)ctx->ev_off.p;
    if (ctx->src_kind == PP_SRC_TRACE32)
        k4_segment_stats<float><<<grid, 256, 0, ctx->stream>>>(
            (const float *)ctx->trace, (const int64_t *)ctx->ev_start.p, ev_off, ctx->ctr, rows_are_events, flat_start,
            row_event, cap_rows, mean, sd, mn, mx, ctx->adc);
    else if (ctx->src_kind == PP_SRC_ADC16)
        k4_segment_stats<int16_t><<<grid, 256, 0, ctx->stream>>>(
            (const int16_t *)ctx->trace, (const int64_t *)ctx->ev_start.p, ev_off, ctx->ctr, rows_are_events, flat_start,
            row_event, cap_rows, mean, sd, mn, mx, ctx->adc);
    else
        k4_segment_stats<double><<<grid, 256, 0, ctx->stream>>>(
            f64_samples(ctx), f64_bases(ctx), ev_off, ctx->ctr, rows_are_events, flat_start, row_event, cap_rows,
            mean, sd, mn, mx, ctx->adc);
    LAUNCHED(ctx);
    return PP_OK;
}

int enqueue_stats(pp_ctx *ctx)
{
    StageRange nvtx_range("pypore:stats");
    CKR(launch_stats(ctx, 0, (const int64_t *)ctx->seg_flat.p, (const int *)ctx->seg_event.p, ctx->cap_segs,
                     (double *)ctx->seg_mean.p, (double *)ctx->seg_std.p, (double *)ctx->seg_min.p,
                     (double *)ctx->seg_max.p));
    CKR(end_stage(ctx, ST_STATS));
    ctx->stats_valid = true;
    return PP_OK;
}

int check_overflow(pp_ctx *ctx)
{
    const unsigned o = ctx->h_ctr->overflow;
    if (o & PP_OVF_QUEUE) return fail(ctx, PP_ERR_CAPACITY, "split work queue overflow");
    if (o & PP_OVF_SEGS) return fail(ctx, PP_ERR_CAPACITY, "segment table overflow");
    if (o & PP_OVF_FILTER_SHORT)
        return fail(ctx, PP_ERR_FILTER_LEN,
                    "The length of the input vector x must be greater than padlen");
    return PP_OK;
}

void absorb_counters(pp_ctx *ctx)
{
    const PPCounters *h = ctx->h_ctr;
    ctx->n_events = (int64_t)h->n_events;
    ctx->n_event_samples = (int64_t)h->n_event_samples;
    ctx->split_counters[0] = (int64_t)h->n_cand;
    ctx->split_counters[1] = (int64_t)h->n_scan;
    ctx->split_counters[2] = (int64_t)h->n_seq_redo;
    ctx->split_counters[3] = (int64_t)h->n_tasks;
    ctx->split_counters[4] = (int64_t)h->n_exact;
    ctx->split_counters[5] = (int64_t)h->n_sure;
    ctx->split_counters[6] = (int64_t)h->n_multi;
    ctx->split_counters[7] = (int64_t)h->n_full;
}

// End of a pipeline call, counters fetched: the table sizes the device counted, out = runs, events, event samples,
// segments
int commit_counters(pp_ctx *ctx, int64_t out[4])
{
    absorb_counters(ctx);
    CKR(check_overflow(ctx));
    ctx->n_segments = (int64_t)ctx->h_ctr->n_segments;
    if (out) {
        out[0] = ctx->n_runs;
        out[1] = ctx->n_events;
        out[2] = ctx->n_event_samples;
        out[3] = ctx->n_segments;
    }
    return PP_OK;
}

// Enqueue a call that begins with a threshold scan, then fetch the counters; a run table that overflowed is regrown
// to what the scan counted and the call repeats once
template <typename Enqueue>
int with_run_retry(pp_ctx *ctx, Enqueue enqueue)
{
    for (int attempt = 0; attempt < 2; ++attempt) {
        CKR(enqueue());
        CKR(fetch_counters(ctx));
        const int64_t runs = (int64_t)ctx->h_ctr->n_runs;
        if (runs <= ctx->cap_runs) {
            ctx->n_runs = runs;
            return PP_OK;
        }
        CKR(ensure_run_buffers(ctx, runs + 16));
    }
    return fail(ctx, PP_ERR_CAPACITY, "run table overflow");
}

// Copy the rows not exported yet to the host tables and wait for them; tables too small for every row fail with
// PP_ERR_CAPACITY (the device tables stay whole)
int export_tables(pp_ctx *ctx, const PPHostTables &H, int with_stats)
{
    CKR(enqueue_export(ctx, H, with_stats));
    CKR(fetch_counters(ctx));
    if (ctx->h_ctr->overflow & PP_OVF_EXPORT) return fail(ctx, PP_ERR_CAPACITY, "host tables too small");
    return PP_OK;
}

}  // namespace

// ===========================================================================
extern "C" {

int pp_version(void) { return 100; }

int pp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int pp_create(int device, void *cuda_stream, pp_ctx **out)
{
    if (!out) return PP_ERR_ARG;
    *out = nullptr;
    pp_ctx *ctx = new (std::nothrow) pp_ctx();
    if (!ctx) return PP_ERR_ARG;
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { delete ctx; return PP_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return PP_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    if (prop.major < 10) {
        // sm_100a-only binary: fail loudly instead of a cryptic launch error
        delete ctx;
        return PP_ERR_CUDA;
    }
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return PP_ERR_CUDA;
        }
        ctx->own_stream = true;
    }
    bool ok = cudaMalloc((void **)&ctx->ctr, sizeof(PPCounters)) == cudaSuccess &&
              cudaMallocHost((void **)&ctx->h_ctr, sizeof(PPCounters)) == cudaSuccess &&
              cudaMemset(ctx->ctr, 0, sizeof(PPCounters)) == cudaSuccess;
    for (int i = 0; ok && i <= ST_COUNT; ++i) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k3_split, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)K3_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k3_flow, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)K3F_SMEM_BYTES) == cudaSuccess;
    if (!ok) { pp_destroy(ctx); return PP_ERR_CUDA; }
    memset(ctx->h_ctr, 0, sizeof(PPCounters));
    *out = ctx;
    return PP_OK;
}

void pp_destroy(pp_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int q = 0; q < 64; ++q)
        if (ctx->ctl_ipc[q] && ctx->ctl_peers[q]) cudaIpcCloseMemHandle(ctx->ctl_peers[q]);
    if (ctx->ctr) cudaFree(ctx->ctr);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    for (int i = 0; i <= ST_COUNT; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->copy_ev) cudaEventDestroy(ctx->copy_ev);
    if (ctx->compute_ev) cudaEventDestroy(ctx->compute_ev);
    if (ctx->pf_t0) cudaEventDestroy(ctx->pf_t0);
    if (ctx->pf_t1) cudaEventDestroy(ctx->pf_t1);
    for (auto &q : ctx->pend) {
        if (q.done) cudaEventDestroy(q.done);
        if (q.t0) cudaEventDestroy(q.t0);
        if (q.t1) cudaEventDestroy(q.t1);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;   // the device buffers free themselves
}

const char *pp_last_error(pp_ctx *ctx) { return ctx ? ctx->err : "null context"; }

void *pp_stream(pp_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int pp_host_alloc(pp_ctx *ctx, int64_t bytes, void **out)
{
    if (!ctx || !out || bytes <= 0) return fail(ctx, PP_ERR_ARG, "bad host allocation");
    CKR(set_device(ctx));
    CK(cudaMallocHost(out, (size_t)bytes));
    return PP_OK;
}

void pp_host_free(pp_ctx *ctx, void *p)
{
    if (ctx) cudaSetDevice(ctx->device);
    if (p) cudaFreeHost(p);
}

int pp_sync(pp_ctx *ctx)
{
    if (!ctx) return PP_ERR_ARG;
    CKR(set_device(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_set_option(pp_ctx *ctx, int option, int64_t value)
{
    if (!ctx) return PP_ERR_ARG;
    switch (option) {
    case PP_OPT_SCREEN: ctx->opt_screen = value ? 1 : 0; return PP_OK;
    case PP_OPT_SPINE: ctx->opt_spine = value ? 1 : 0; return PP_OK;
    case PP_OPT_SPLIT_KERNEL: ctx->opt_split_kernel = value ? 1 : 0; return PP_OK;
    case PP_OPT_SPLIT_CTAS:
        if (value < 0 || value > (1 << 20)) return fail(ctx, PP_ERR_ARG, "bad CTA count %lld", (long long)value);
        ctx->opt_split_ctas = (int)value;
        return PP_OK;
    default: return fail(ctx, PP_ERR_ARG, "unknown option %d", option);
    }
}

int pp_get_option(pp_ctx *ctx, int option, int64_t *value)
{
    if (!ctx || !value) return PP_ERR_ARG;
    switch (option) {
    case PP_OPT_SCREEN: *value = ctx->opt_screen; return PP_OK;
    case PP_OPT_SPINE: *value = ctx->opt_spine; return PP_OK;
    case PP_OPT_SPLIT_KERNEL: *value = ctx->opt_split_kernel; return PP_OK;
    case PP_OPT_SPLIT_CTAS: *value = ctx->opt_split_ctas; return PP_OK;
    default: return fail(ctx, PP_ERR_ARG, "unknown option %d", option);
    }
}

int64_t pp_launch_count(pp_ctx *ctx) { return ctx ? ctx->launches : 0; }

int pp_stage_ms(pp_ctx *ctx, int stage, float *ms)
{
    if (!ctx || !ms || stage < 0 || stage >= ST_COUNT) return PP_ERR_ARG;
    *ms = 0.f;
    if (!ctx->stage_ran[stage] || !ctx->rec[stage + 1]) return PP_OK;
    int prev = stage;  // nearest recorded boundary at or before the stage's start
    while (prev > 0 && !ctx->rec[prev]) --prev;
    if (!ctx->rec[prev]) return PP_OK;
    CK(cudaEventElapsedTime(ms, ctx->ev[prev], ctx->ev[stage + 1]));
    return PP_OK;
}

// ---- trace ------------------------------------------------------------------
static int trace_upload_impl(pp_ctx *ctx, const void *host, int64_t n, int64_t extra_capacity, int kind)
{
    if (!ctx || !host || n <= 0 || extra_capacity < 0) return fail(ctx, PP_ERR_ARG, "bad trace");
    const size_t elem = sample_bytes(kind);
    CKR(set_device(ctx));
    CKR(ensure(ctx, ctx->trace_buf, elem * (size_t)(n + extra_capacity)));
    CK(cudaMemcpyAsync(ctx->trace_buf.p, host, elem * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    set_trace(ctx, ctx->trace_buf.p, kind, n, (int64_t)(ctx->trace_buf.cap / elem));
    return PP_OK;
}

int pp_trace_upload(pp_ctx *ctx, const float *host, int64_t n, int64_t extra_capacity)
{
    return trace_upload_impl(ctx, host, n, extra_capacity, PP_SRC_TRACE32);
}

int pp_trace_upload_f64(pp_ctx *ctx, const double *host, int64_t n)
{
    return trace_upload_impl(ctx, host, n, 0, PP_SRC_TRACE64);
}

// decode(c) on the host: the product is rounded on its own (no contraction into an FMA), like the device's
static double adc_decode_host(int c, double scale, double offset)
{
    volatile double prod = (double)c * scale;
    return prod + offset;
}

int pp_adc16_check(double scale, double offset)
{
    if (!isfinite(scale) || scale == 0.0 || !isfinite(offset)) return PP_ERR_ARG;
    // decode is monotone in c: every count decodes to a finite value iff both ends do
    if (!isfinite(adc_decode_host(-32768, scale, offset)) || !isfinite(adc_decode_host(32767, scale, offset)))
        return PP_ERR_ARG;
    return PP_OK;
}

int pp_adc16_key_threshold(double scale, double offset, double threshold, int32_t *key, int32_t *kxor)
{
    if (!key || !kxor || pp_adc16_check(scale, offset) != PP_OK) return PP_ERR_ARG;
    // decode(k ^ kx) is non-decreasing in the key k, so `!(decode < threshold)` is false, then true over the 65,536
    // keys (true throughout for a NaN threshold): find the first key where it holds, 32768 if none does
    const int kx = scale < 0.0 ? -1 : 0;
    int lo = -32768, hi = 32768;
    while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);
        if (!(adc_decode_host(mid ^ kx, scale, offset) < threshold)) hi = mid;
        else lo = mid + 1;
    }
    *key = lo;
    *kxor = kx;
    return PP_OK;
}

int pp_trace_upload_adc16(pp_ctx *ctx, const int16_t *host, int64_t n, double scale, double offset)
{
    if (pp_adc16_check(scale, offset) != PP_OK)
        return fail(ctx, PP_ERR_ARG, "ADC scale must be finite and non-zero, offset finite, every count decoding finite");
    CKR(trace_upload_impl(ctx, host, n, 0, PP_SRC_ADC16));
    ctx->adc = PPAdc{scale, offset};
    return PP_OK;
}

// ---- double-buffered upload (back-to-back traces: the copy of trace i+1 runs under the kernels of trace i) ----
static int ensure_copy_stream(pp_ctx *ctx)
{
    if (!ctx->copy_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->copy_ev, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->compute_ev, cudaEventDisableTiming));
    }
    return PP_OK;
}

int pp_trace_prefetch(pp_ctx *ctx, const float *host, int64_t n, int64_t extra_capacity)
{
    if (!ctx || !host || n <= 0 || extra_capacity < 0) return fail(ctx, PP_ERR_ARG, "bad trace");
    CKR(require_trace(ctx, NOT_ADC, "prefetch takes float32 traces"));
    if (ctx->n_pend >= 2) return fail(ctx, PP_ERR_STATE, "two prefetched traces are already waiting for pp_trace_swap");
    CKR(set_device(ctx));
    CKR(ensure_copy_stream(ctx));
    pp_ctx::Pending &q = ctx->pend[ctx->n_pend];
    if (!q.done) {
        CK(cudaEventCreateWithFlags(&q.done, cudaEventDisableTiming));
        CK(cudaEventCreate(&q.t0));
        CK(cudaEventCreate(&q.t1));
    }
    if (!q.buf.p) q.buf = std::move(ctx->trace_spare);     // the buffer the last swap retired, if any
    CKR(ensure(ctx, q.buf, sizeof(float) * (size_t)(n + extra_capacity)));
    // the buffer was the resident trace some swaps ago: whatever still reads it was enqueued before this point
    CK(cudaEventRecord(ctx->compute_ev, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->compute_ev, 0));
    CK(cudaEventRecord(q.t0, ctx->copy_stream));
    CK(cudaMemcpyAsync(q.buf.p, host, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream));
    CK(cudaEventRecord(q.t1, ctx->copy_stream));
    CK(cudaEventRecord(q.done, ctx->copy_stream));
    q.n = n;
    ++ctx->n_pend;
    return PP_OK;
}

int pp_trace_prefetch_ms(pp_ctx *ctx, float *ms)
{
    if (!ctx || !ms) return PP_ERR_ARG;
    if (!ctx->pf_t1) return fail(ctx, PP_ERR_STATE, "no prefetched trace has been swapped in so far");
    CKR(set_device(ctx));
    CK(cudaEventSynchronize(ctx->pf_t1));
    CK(cudaEventElapsedTime(ms, ctx->pf_t0, ctx->pf_t1));
    return PP_OK;
}

int pp_trace_swap(pp_ctx *ctx)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_pend <= 0) return fail(ctx, PP_ERR_STATE, "no prefetched trace");
    CKR(set_device(ctx));
    pp_ctx::Pending &q = ctx->pend[0];
    CK(cudaStreamWaitEvent(ctx->stream, q.done, 0));   // stream-level: the host goes on
    // the retired resident buffer becomes the spare one (an older spare is dropped: at most three buffers live)
    ctx->trace_spare = std::move(ctx->trace_buf);
    ctx->trace_buf = std::move(q.buf);
    // the timing events of the trace swapped in are what pp_trace_prefetch_ms reads
    cudaEvent_t a = ctx->pf_t0, b = ctx->pf_t1;
    ctx->pf_t0 = q.t0; ctx->pf_t1 = q.t1;
    q.t0 = a; q.t1 = b;
    if (!q.t0) { CK(cudaEventCreate(&q.t0)); CK(cudaEventCreate(&q.t1)); }
    set_trace(ctx, ctx->trace_buf.p, PP_SRC_TRACE32, q.n, (int64_t)(ctx->trace_buf.cap / sizeof(float)));
    q.n = -1;
    if (ctx->n_pend == 2) std::swap(ctx->pend[0], ctx->pend[1]);   // the younger one moves up
    --ctx->n_pend;
    return PP_OK;
}

int pp_trace_adopt(pp_ctx *ctx, const float *dev, int64_t n, int64_t capacity)
{
    if (!ctx || !dev || n <= 0 || capacity < n) return fail(ctx, PP_ERR_ARG, "bad trace");
    if (((uintptr_t)dev) & 15) return fail(ctx, PP_ERR_ARG, "device trace must be 16-byte aligned");
    CKR(require_trace(ctx, NOT_ADC, "adopt takes float32 traces"));
    set_trace(ctx, dev, PP_SRC_TRACE32, n, capacity);
    return PP_OK;
}

int pp_trace_append(pp_ctx *ctx, const float *src, int64_t n, int src_is_device)
{
    if (!ctx || !src || n < 0) return fail(ctx, PP_ERR_ARG, "bad append");
    CKR(require_trace(ctx, TAKES_F32, "append takes float32 traces"));
    if (ctx->n + n > ctx->trace_cap) return fail(ctx, PP_ERR_CAPACITY, "trace capacity exceeded");
    CKR(set_device(ctx));
    CK(cudaMemcpyAsync((float *)ctx->trace + ctx->n, src, sizeof(float) * (size_t)n,
                       src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    ctx->n += n;
    return PP_OK;
}

int pp_trace_truncate(pp_ctx *ctx, int64_t n)
{
    if (!ctx || n <= 0 || n > ctx->n) return fail(ctx, PP_ERR_ARG, "bad truncate");
    ctx->n = n;
    return PP_OK;
}

int pp_trace_extend(pp_ctx *ctx, int64_t n)
{
    if (!ctx || n < 0) return fail(ctx, PP_ERR_ARG, "bad extend");
    CKR(require_trace(ctx, TAKES_F32, "extend takes float32 traces"));
    if (ctx->n + n > ctx->trace_cap) return fail(ctx, PP_ERR_CAPACITY, "trace capacity exceeded");
    ctx->n += n;
    return PP_OK;
}

int64_t pp_trace_len(pp_ctx *ctx) { return ctx ? ctx->n : 0; }
const float *pp_trace_device_ptr(pp_ctx *ctx) { return ctx ? trace_as<float>(ctx, PP_SRC_TRACE32) : nullptr; }

// ---- K1 -----------------------------------------------------------------------
int pp_threshold_scan(pp_ctx *ctx, double threshold, int64_t scan_len, int64_t *n_runs)
{
    if (!ctx) return PP_ERR_ARG;
    CKR(with_run_retry(ctx, [&]() -> int {
        CKR(begin_call(ctx, 0));
        CKR(enqueue_threshold(ctx, threshold, scan_len));
        return end_stage(ctx, ST_THRESHOLD);
    }));
    if (n_runs) *n_runs = ctx->n_runs;
    return PP_OK;
}

int pp_runs_download(pp_ctx *ctx, int64_t cap, int64_t *start, int64_t *length, double *mn,
                     double *mx, uint8_t *below)
{
    if (!ctx) return PP_ERR_ARG;
    if (cap < ctx->n_runs) return fail(ctx, PP_ERR_CAPACITY, "run buffers too small");
    return pp_runs_download_range(ctx, 0, ctx->n_runs, start, length, mn, mx, below);
}

int pp_runs_download_range(pp_ctx *ctx, int64_t first, int64_t count, int64_t *start, int64_t *length,
                           double *mn, double *mx, uint8_t *below)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_runs < 0) return fail(ctx, PP_ERR_STATE, "pp_threshold_scan has not run");
    if (first < 0 || count < 0 || first + count > ctx->n_runs) return fail(ctx, PP_ERR_ARG, "bad run range");
    CKR(set_device(ctx));
    const size_t r = (size_t)count, o = (size_t)first;
    if (r) {
        if (start) CK(cudaMemcpyAsync(start, (int64_t *)ctx->run_start.p + o, 8 * r, cudaMemcpyDeviceToHost, ctx->stream));
        if (length) CK(cudaMemcpyAsync(length, (int64_t *)ctx->run_len.p + o, 8 * r, cudaMemcpyDeviceToHost, ctx->stream));
        if (mn) CK(cudaMemcpyAsync(mn, (double *)ctx->run_min.p + o, 8 * r, cudaMemcpyDeviceToHost, ctx->stream));
        if (mx) CK(cudaMemcpyAsync(mx, (double *)ctx->run_max.p + o, 8 * r, cudaMemcpyDeviceToHost, ctx->stream));
        if (below) CK(cudaMemcpyAsync(below, (unsigned char *)ctx->run_below.p + o, r, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_select_events(pp_ctx *ctx, int rule_mask, int64_t duration_gt, int64_t duration_lt,
                     double min_gt, double max_lt, int skip_first, int skip_last, int64_t *n_events,
                     int64_t *n_event_samples)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_runs < 0) return fail(ctx, PP_ERR_STATE, "pp_threshold_scan has not run");
    CKR(set_device(ctx));
    CKR(enqueue_select(ctx, rule_mask, duration_gt, duration_lt, min_gt, max_lt, skip_first, skip_last));
    CKR(end_stage(ctx, ST_SELECT));
    CKR(fetch_counters(ctx));
    absorb_counters(ctx);
    if (n_events) *n_events = ctx->n_events;
    if (n_event_samples) *n_event_samples = ctx->n_event_samples;
    return PP_OK;
}

int pp_set_events(pp_ctx *ctx, const int64_t *start, const int64_t *length, int64_t n_events)
{
    if (!ctx || n_events < 0 || (n_events > 0 && (!start || !length)))
        return fail(ctx, PP_ERR_ARG, "bad events");
    if (!ctx->trace) return fail(ctx, PP_ERR_STATE, "no trace resident");
    CKR(set_device(ctx));
    for (int64_t i = 0; i < n_events; ++i)
        if (start[i] < 0 || length[i] <= 0 || start[i] + length[i] > ctx->n)
            return fail(ctx, PP_ERR_ARG, "event %lld out of range", (long long)i);
    CKR(ensure_event_buffers(ctx, n_events + 16));
    if (n_events) {
        CK(cudaMemcpyAsync(ctx->ev_start.p, start, 8 * (size_t)n_events, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->ev_len.p, length, 8 * (size_t)n_events, cudaMemcpyHostToDevice, ctx->stream));
    }
    k1_event_offsets<<<1, SEL_THREADS, 0, ctx->stream>>>(ctx->ctr, (const int64_t *)ctx->ev_len.p, n_events,
                                                         (int64_t *)ctx->ev_off.p);
    LAUNCHED(ctx);
    ctx->src_kind = ctx->trace_kind;
    int64_t tot = 0;
    for (int64_t i = 0; i < n_events; ++i) tot += length[i];
    ctx->flat_cap = tot > 0 ? tot : 1;
    CK(cudaStreamSynchronize(ctx->stream));  // host arrays may be freed by the caller
    drop_from(ctx, LV_EVENTS);
    ctx->n_events = n_events;
    ctx->n_event_samples = tot;
    return PP_OK;
}

__global__ void k_append_event(PPCounters *ctr, int64_t *ev_start, int64_t *ev_len, int64_t *ev_off,
                               int64_t start, int64_t length)
{
    const unsigned long long e = ctr->n_events;
    ev_start[e] = start;
    ev_len[e] = length;
    // ev_off[e] already holds the running total
    ev_off[e + 1] = ev_off[e] + length;
    ctr->n_events = e + 1;
    ctr->n_event_samples += (unsigned long long)length;
}

int pp_append_event(pp_ctx *ctx, int64_t start, int64_t length)
{
    if (!ctx || start < 0 || length <= 0 || start + length > ctx->n)
        return fail(ctx, PP_ERR_ARG, "bad appended event");
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    CKR(set_device(ctx));
    CKR(ensure_event_buffers(ctx, ctx->n_events + 16));
    k_append_event<<<1, 1, 0, ctx->stream>>>(ctx->ctr, (int64_t *)ctx->ev_start.p, (int64_t *)ctx->ev_len.p,
                                             (int64_t *)ctx->ev_off.p, start, length);
    LAUNCHED(ctx);
    ctx->n_events += 1;
    ctx->n_event_samples += length;
    drop_from(ctx, LV_PREFIX);
    if (ctx->flat_cap < ctx->n) ctx->flat_cap = ctx->n;
    return PP_OK;
}

int pp_events_download(pp_ctx *ctx, int64_t cap, int64_t *start, int64_t *length)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    if (cap < ctx->n_events) return fail(ctx, PP_ERR_CAPACITY, "event buffers too small");
    CKR(set_device(ctx));
    const size_t e = (size_t)ctx->n_events;
    if (start && e) CK(cudaMemcpyAsync(start, ctx->ev_start.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    if (length && e) CK(cudaMemcpyAsync(length, ctx->ev_len.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_events_upload_f64(pp_ctx *ctx, const double *host, const int64_t *length, int64_t n_events)
{
    if (!ctx || !host || !length || n_events <= 0) return fail(ctx, PP_ERR_ARG, "bad events");
    CKR(set_device(ctx));
    int64_t tot = 0;
    for (int64_t i = 0; i < n_events; ++i) {
        if (length[i] <= 0) return fail(ctx, PP_ERR_ARG, "event %lld is empty", (long long)i);
        tot += length[i];
    }
    CKR(ensure_event_buffers(ctx, n_events + 16));
    CKR(ensure(ctx, ctx->flat64, sizeof(double) * (size_t)tot));
    CK(cudaMemcpyAsync(ctx->flat64.p, host, sizeof(double) * (size_t)tot, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->ev_len.p, length, 8 * (size_t)n_events, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->ctr, 0, sizeof(PPCounters), ctx->stream));
    k1_event_offsets<<<1, SEL_THREADS, 0, ctx->stream>>>(ctx->ctr, (const int64_t *)ctx->ev_len.p, n_events,
                                                         (int64_t *)ctx->ev_off.p);
    LAUNCHED(ctx);
    // ev_start mirrors ev_off for a packed source
    CK(cudaMemcpyAsync(ctx->ev_start.p, ctx->ev_off.p, 8 * (size_t)n_events, cudaMemcpyDeviceToDevice,
                       ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->src_kind = PP_SRC_FLAT64;
    ctx->flat_cap = tot;
    drop_from(ctx, LV_EVENTS);
    ctx->n_events = n_events;
    ctx->n_event_samples = tot;
    return PP_OK;
}

// ---- K5 -----------------------------------------------------------------------
int pp_filter_events(pp_ctx *ctx, const double *b, const double *a, const double *zi, int ncoef)
{
    if (!ctx || !b || !a || ncoef < 2 || ncoef > FILT_MAX_COEF || (ncoef > 1 && !zi))
        return fail(ctx, PP_ERR_ARG, "bad filter coefficients");
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    CKR(begin_call(ctx, ST_FILTER));
    CKR(enqueue_filter(ctx, b, a, zi, ncoef));
    CKR(fetch_counters(ctx));
    return check_overflow(ctx);
}

int pp_event_samples_download(pp_ctx *ctx, int64_t cap, double *out)
{
    if (!ctx || !out) return PP_ERR_ARG;
    if (ctx->n_event_samples < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    if (cap < ctx->n_event_samples) return fail(ctx, PP_ERR_CAPACITY, "sample buffer too small");
    CKR(set_device(ctx));
    if (ctx->src_kind != PP_SRC_FLAT64) return fail(ctx, PP_ERR_STATE, "events are views of the trace");
    CK(cudaMemcpyAsync(out, ctx->flat64.p, 8 * (size_t)ctx->n_event_samples, cudaMemcpyDeviceToHost,
                       ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

// ---- K2+K3 --------------------------------------------------------------------
int pp_statsplit(pp_ctx *ctx, int min_width, int max_width, int window_width, double min_gain,
                 int prefix_mode, int64_t *n_segments)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    CKR(begin_call(ctx, ST_PREFIX));
    CKR(enqueue_split(ctx, min_width, max_width, window_width, min_gain, prefix_mode));
    CKR(fetch_counters(ctx));
    CKR(commit_counters(ctx, nullptr));
    if (n_segments) *n_segments = ctx->n_segments;
    return PP_OK;
}

int pp_prefix(pp_ctx *ctx, int prefix_mode)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    CKR(set_device(ctx));
    const int64_t ncap = ctx->flat_cap;
    if (ncap <= 0) return fail(ctx, PP_ERR_STATE, "no events selected");
    CKR(ensure(ctx, ctx->cc, sizeof(double2) * ncap));
    CKR(enqueue_prefix(ctx, prefix_mode));
    CKR(fetch_counters(ctx));
    ctx->split_counters[2] = (int64_t)ctx->h_ctr->n_seq_redo;
    ctx->prefix_valid = true;
    return PP_OK;
}

int pp_window_gains(pp_ctx *ctx, int64_t ev, int n_windows, const int32_t *ps, const int32_t *pe, int min_width,
                    double *out, int64_t cap)
{
    if (!ctx || !ps || !pe || !out || n_windows <= 0 || min_width < 0) return fail(ctx, PP_ERR_ARG, "bad windows");
    if (!ctx->prefix_valid) return fail(ctx, PP_ERR_STATE, "prefix sums are not resident (pp_prefix / pp_statsplit)");
    if (ev < 0 || ev >= ctx->n_events) return fail(ctx, PP_ERR_ARG, "bad event index");
    CKR(set_device(ctx));
    std::vector<int64_t> off;
    CKR(host_scratch(ctx, off, (size_t)n_windows));
    int64_t total = 0;
    for (int w = 0; w < n_windows; ++w) {
        off[w] = total;
        const int64_t n = (int64_t)pe[w] - ps[w] - 2LL * min_width + 1;
        if (ps[w] < 0 || pe[w] < ps[w]) return fail(ctx, PP_ERR_ARG, "bad window %d", w);
        if (n > 0) total += n;
    }
    if (total > cap) return fail(ctx, PP_ERR_CAPACITY, "gain buffer too small");
    DevBuf d_ps, d_pe, d_off, d_out;
    CKR(ensure(ctx, d_ps, 4 * (size_t)n_windows));
    CKR(ensure(ctx, d_pe, 4 * (size_t)n_windows));
    CKR(ensure(ctx, d_off, 8 * (size_t)n_windows));
    CKR(ensure(ctx, d_out, 8 * (size_t)(total > 0 ? total : 1)));
    CK(cudaMemcpyAsync(d_ps.p, ps, 4 * (size_t)n_windows, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_pe.p, pe, 4 * (size_t)n_windows, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_off.p, off.data(), 8 * (size_t)n_windows, cudaMemcpyHostToDevice, ctx->stream));
    K3Global G;
    memset(&G, 0, sizeof G);
    G.cc = (const double2 *)ctx->cc.p;
    G.ev_off = (const int64_t *)ctx->ev_off.p;
    const dim3 grid(32, n_windows < 4096 ? n_windows : 4096);
    k3_window_gains<<<grid, 256, 0, ctx->stream>>>(G, (int)ev, n_windows, (const int *)d_ps.p, (const int *)d_pe.p,
                                                   min_width, (const int64_t *)d_off.p, (double *)d_out.p);
    LAUNCHED(ctx);
    if (total > 0) CK(cudaMemcpyAsync(out, d_out.p, 8 * (size_t)total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_segment_stats(pp_ctx *ctx)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_segments < 0) return fail(ctx, PP_ERR_STATE, "pp_statsplit has not run");
    CKR(begin_call(ctx, ST_STATS));
    return enqueue_stats(ctx);
}

int pp_segments_download(pp_ctx *ctx, int64_t cap, int32_t *event, int64_t *start, int64_t *end,
                         double *mean, double *std, double *mn, double *mx)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_segments < 0) return fail(ctx, PP_ERR_STATE, "pp_statsplit has not run");
    if (cap < ctx->n_segments) return fail(ctx, PP_ERR_CAPACITY, "segment buffers too small");
    if ((mean || std || mn || mx) && !ctx->stats_valid)
        return fail(ctx, PP_ERR_STATE, "pp_segment_stats has not run");
    CKR(set_device(ctx));
    const size_t s = (size_t)ctx->n_segments;
    if (s) {
        if (event) CK(cudaMemcpyAsync(event, ctx->seg_event.p, 4 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (start) CK(cudaMemcpyAsync(start, ctx->seg_start.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (end) CK(cudaMemcpyAsync(end, ctx->seg_end.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (mean) CK(cudaMemcpyAsync(mean, ctx->seg_mean.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (std) CK(cudaMemcpyAsync(std, ctx->seg_std.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (mn) CK(cudaMemcpyAsync(mn, ctx->seg_min.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
        if (mx) CK(cudaMemcpyAsync(mx, ctx->seg_max.p, 8 * s, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_event_stats_download(pp_ctx *ctx, int64_t cap, double *mean, double *std, double *mn, double *mx)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->n_events < 0) return fail(ctx, PP_ERR_STATE, "no event table");
    if (cap < ctx->n_events) return fail(ctx, PP_ERR_CAPACITY, "event buffers too small");
    CKR(set_device(ctx));
    const size_t e = (size_t)ctx->n_events;
    if (!e) return PP_OK;
    CKR(ensure(ctx, ctx->evs_mean, 8 * e));
    CKR(ensure(ctx, ctx->evs_std, 8 * e));
    CKR(ensure(ctx, ctx->evs_min, 8 * e));
    CKR(ensure(ctx, ctx->evs_max, 8 * e));
    CKR(launch_stats(ctx, 1, (const int64_t *)ctx->ev_off.p, nullptr, (int64_t)e, (double *)ctx->evs_mean.p,
                     (double *)ctx->evs_std.p, (double *)ctx->evs_min.p, (double *)ctx->evs_max.p));
    if (mean) CK(cudaMemcpyAsync(mean, ctx->evs_mean.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    if (std) CK(cudaMemcpyAsync(std, ctx->evs_std.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    if (mn) CK(cudaMemcpyAsync(mn, ctx->evs_min.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    if (mx) CK(cudaMemcpyAsync(mx, ctx->evs_max.p, 8 * e, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

const void *pp_table_device_ptr(pp_ctx *ctx, int which)
{
    if (!ctx) return nullptr;
    switch (which) {
    case 0: return ctx->seg_event.p;
    case 1: return ctx->seg_start.p;
    case 2: return ctx->seg_end.p;
    case 3: return ctx->seg_mean.p;
    case 4: return ctx->seg_std.p;
    case 5: return ctx->seg_min.p;
    case 6: return ctx->seg_max.p;
    case 7: return ctx->ev_start.p;
    case 8: return ctx->ev_len.p;
    default: return nullptr;
    }
}

int pp_split_counters(pp_ctx *ctx, int64_t out[8])
{
    if (!ctx || !out) return PP_ERR_ARG;
    for (int i = 0; i < 8; ++i) out[i] = ctx->split_counters[i];
    return PP_OK;
}

int pp_debug_screen(pp_ctx *ctx, int64_t ev, int ps, int pe, int min_width, double *h_screen,
                    double *h_exact, uint8_t *ok, double *eps)
{
    if (!ctx || !h_screen || !h_exact || !ok) return PP_ERR_ARG;
    if (ctx->n_segments < 0) return fail(ctx, PP_ERR_STATE, "pp_statsplit has not run");
    const int n = pe - ps - 2 * min_width + 1;
    if (ev < 0 || ev >= ctx->n_events || ps < 0 || n <= 0 || pe - ps + 1 > ctx->T_len)
        return fail(ctx, PP_ERR_ARG, "bad debug window");
    CKR(set_device(ctx));
    DevBuf a, b, c;
    CKR(ensure(ctx, a, 8 * (size_t)n));
    CKR(ensure(ctx, b, 8 * (size_t)n));
    CKR(ensure(ctx, c, (size_t)n));
    K3Global G;
    memset(&G, 0, sizeof G);
    G.cc = (const double2 *)ctx->cc.p;
    G.ev_off = (const int64_t *)ctx->ev_off.p;
    G.RN = (const double *)ctx->Ttab.p;
    k3_debug_screen<<<64, 256, 0, ctx->stream>>>(G, (int)ev, ps, pe, min_width, (double *)a.p, (double *)b.p,
                                                 (unsigned char *)c.p);
    LAUNCHED(ctx);
    CK(cudaMemcpyAsync(h_screen, a.p, 8 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_exact, b.p, 8 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ok, c.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (eps) *eps = (double)(pe - ps) * K3_EPS_PER_SAMPLE + K3_EPS_CONST;
    return PP_OK;
}

int pp_debug_prefix(pp_ctx *ctx, int64_t cap, double *c, double *c2, uint8_t *redone)
{
    if (!ctx || !c || !c2 || !redone) return PP_ERR_ARG;
    if (!ctx->prefix_valid) return fail(ctx, PP_ERR_STATE, "prefix sums are not resident (pp_prefix / pp_statsplit)");
    if (cap < ctx->n_event_samples || cap < ctx->n_events) return fail(ctx, PP_ERR_CAPACITY, "buffers too small");
    CKR(set_device(ctx));
    const size_t n = (size_t)ctx->n_event_samples, e = (size_t)ctx->n_events;
    std::vector<double2> cc;
    std::vector<unsigned> fl;
    CKR(host_scratch(ctx, cc, n));
    CKR(host_scratch(ctx, fl, e));
    if (n) CK(cudaMemcpyAsync(cc.data(), ctx->cc.p, sizeof(double2) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (e && ctx->prefix_mode == PP_PREFIX_AUTO)
        CK(cudaMemcpyAsync(fl.data(), ctx->inexact.p, sizeof(unsigned) * e, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; ++i) { c[i] = cc[i].x; c2[i] = cc[i].y; }
    // PARALLEL redoes nothing, SEQUENTIAL runs every event in the strict order
    for (size_t i = 0; i < e; ++i)
        redone[i] = ctx->prefix_mode == PP_PREFIX_AUTO ? (fl[i] != 0u) : ctx->prefix_mode == PP_PREFIX_SEQUENTIAL;
    return PP_OK;
}

int pp_debug_lg2_error(pp_ctx *ctx, double *max_err)
{
    if (!ctx || !max_err) return PP_ERR_ARG;
    CKR(set_device(ctx));
    DevBuf a;
    CKR(ensure(ctx, a, 256));
    CK(cudaMemsetAsync(a.p, 0, 8, ctx->stream));
    k3_debug_lg2_error<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>((unsigned long long *)a.p);
    LAUNCHED(ctx);
    CK(cudaMemcpyAsync(max_err, a.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

// ---- pipeline -----------------------------------------------------------------
int pp_pipeline(pp_ctx *ctx, const pp_pipeline_params *p, int64_t out[4])
{
    if (!ctx || !p) return PP_ERR_ARG;
    CKR(with_run_retry(ctx, [&]() -> int {
        CKR(begin_call(ctx, 0));
        CKR(enqueue_threshold(ctx, p->threshold, -1));
        CKR(end_stage(ctx, ST_THRESHOLD));
        CKR(enqueue_select(ctx, p->rule_mask, p->duration_gt, p->duration_lt, p->min_gt, p->max_lt, 0, 0));
        CKR(end_stage(ctx, ST_SELECT));
        if (p->filter_ncoef > 0)
            CKR(enqueue_filter(ctx, p->filter_b, p->filter_a, p->filter_zi, p->filter_ncoef));
        CKR(enqueue_split(ctx, p->min_width, p->max_width, p->window_width, p->min_gain, p->prefix_mode));
        if (p->with_stats) CKR(enqueue_stats(ctx));
        return PP_OK;
    }));
    return commit_counters(ctx, out);
}

// ---- multi-GPU (one context per rank; pypore_b200/dist.py drives the exchange) ------------
int pp_shard_scan(pp_ctx *ctx, double threshold, int64_t scan_len, double *dev_record)
{
    if (!ctx || !dev_record) return PP_ERR_ARG;
    CKR(require_trace(ctx, NOT_ADC, "the sharded path takes float32 traces"));
    CKR(begin_call(ctx, 0));
    CKR(enqueue_threshold(ctx, threshold, scan_len));
    CKR(end_stage(ctx, ST_THRESHOLD));
    k1_boundary_record<<<1, 32, 0, ctx->stream>>>(
        ctx->scan_len, ctx->ctr, (const int64_t *)ctx->run_start.p, (const int64_t *)ctx->run_len.p,
        (const double *)ctx->run_min.p, (const double *)ctx->run_max.p, (const unsigned char *)ctx->run_below.p,
        ctx->cap_runs, dev_record);
    LAUNCHED(ctx);
    return PP_OK;
}

int pp_shard_finish(pp_ctx *ctx, const pp_pipeline_params *p, int skip_first, int skip_last, int has_event,
                    int64_t ev_start, int64_t ev_len, int64_t *dev_record)
{
    if (!ctx || !p || !dev_record) return PP_ERR_ARG;
    CKR(require_trace(ctx, NOT_ADC, "the sharded path takes float32 traces"));
    if (p->filter_ncoef > 0) return fail(ctx, PP_ERR_ARG, "the sharded path does not filter");
    CKR(set_device(ctx));
    CKR(enqueue_select(ctx, p->rule_mask, p->duration_gt, p->duration_lt, p->min_gt, p->max_lt, skip_first,
                       skip_last));
    if (has_event) {
        if (ev_start < 0 || ev_len <= 0 || ev_start + ev_len > ctx->n)
            return fail(ctx, PP_ERR_ARG, "bad appended event");
        k_append_event<<<1, 1, 0, ctx->stream>>>(ctx->ctr, (int64_t *)ctx->ev_start.p, (int64_t *)ctx->ev_len.p,
                                                 (int64_t *)ctx->ev_off.p, ev_start, ev_len);
        LAUNCHED(ctx);
    }
    CKR(end_stage(ctx, ST_SELECT));
    CKR(enqueue_split(ctx, p->min_width, p->max_width, p->window_width, p->min_gain, p->prefix_mode));
    if (p->with_stats) CKR(enqueue_stats(ctx));
    k_result_record<<<1, 32, 0, ctx->stream>>>(ctx->ctr, (long long *)dev_record);
    LAUNCHED(ctx);
    return PP_OK;
}

int pp_shard_plan(pp_ctx *ctx, const double *dev_infos, int rank, int world, const pp_pipeline_params *p,
                  int64_t halo_avail, int64_t *dev_plan)
{
    if (!ctx || !p || !dev_infos || !dev_plan || world < 1 || rank < 0 || rank >= world || halo_avail < 0)
        return fail(ctx, PP_ERR_ARG, "bad shard plan arguments");
    CKR(require_trace(ctx, NOT_ADC, "the sharded path takes float32 traces"));
    CKR(set_device(ctx));
    k_shard_plan<<<1, 32, 0, ctx->stream>>>(dev_infos, rank, world, p->rule_mask, p->duration_gt, p->duration_lt,
                                            p->min_gt, p->max_lt, halo_avail, (long long *)dev_plan);
    LAUNCHED(ctx);
    return PP_OK;
}

int pp_shard_finish_planned(pp_ctx *ctx, const pp_pipeline_params *p, const int64_t *dev_plan, int64_t *dev_record)
{
    if (!ctx || !p || !dev_plan || !dev_record) return PP_ERR_ARG;
    CKR(require_trace(ctx, NOT_ADC, "the sharded path takes float32 traces"));
    if (p->filter_ncoef > 0) return fail(ctx, PP_ERR_ARG, "the sharded path does not filter");
    CKR(set_device(ctx));
    CKR(enqueue_select(ctx, p->rule_mask, p->duration_gt, p->duration_lt, p->min_gt, p->max_lt, 0, 0, 0,
                       (const long long *)dev_plan));
    k_append_planned_event<<<1, 32, 0, ctx->stream>>>(ctx->ctr, (int64_t *)ctx->ev_start.p, (int64_t *)ctx->ev_len.p,
                                                      (int64_t *)ctx->ev_off.p, ctx->cap_events,
                                                      (const long long *)dev_plan);
    LAUNCHED(ctx);
    CKR(end_stage(ctx, ST_SELECT));
    CKR(enqueue_split(ctx, p->min_width, p->max_width, p->window_width, p->min_gain, p->prefix_mode));
    if (p->with_stats) CKR(enqueue_stats(ctx));
    k_result_record<<<1, 32, 0, ctx->stream>>>(ctx->ctr, (long long *)dev_record, (const long long *)dev_plan);
    LAUNCHED(ctx);
    return PP_OK;
}

int pp_shard_commit(pp_ctx *ctx, const int64_t rec[8])
{
    if (!ctx || !rec) return PP_ERR_ARG;
    CKR(require_trace(ctx, NOT_ADC, "the sharded path takes float32 traces"));
    ctx->n_runs = rec[0];
    ctx->n_events = rec[1];
    ctx->n_event_samples = rec[2];
    ctx->n_segments = rec[3];
    ctx->split_counters[0] = rec[5];
    ctx->split_counters[1] = rec[6];
    ctx->split_counters[4] = rec[7];
    const unsigned o = (unsigned)rec[4];
    if (o & PP_OVF_CTL) return fail(ctx, PP_ERR_STATE, "a peer's control record did not arrive (pp_ctl_exchange timed out)");
    if (rec[0] > ctx->cap_runs) return fail(ctx, PP_ERR_CAPACITY, "run table overflow");
    if (o & PP_OVF_QUEUE) return fail(ctx, PP_ERR_CAPACITY, "split work queue overflow");
    if (o & PP_OVF_SEGS) return fail(ctx, PP_ERR_CAPACITY, "segment table overflow");
    return PP_OK;
}

int pp_pack_tables(pp_ctx *ctx, const int64_t *dev_records, int rank, int64_t sample_offset, int64_t *dev_out,
                   int64_t cap_words)
{
    if (!ctx || !dev_out || !dev_records || rank < 0) return PP_ERR_ARG;
    // min / max travel as float32: exact only for segments of a float32 trace's own samples
    if (ctx->src_kind != PP_SRC_TRACE32)
        return fail(ctx, PP_ERR_STATE, "packed tables hold float32 extrema; the segments are not of a float32 trace");
    CKR(set_device(ctx));
    k_pack_tables<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(
        (const long long *)dev_records, rank, cap_words, sample_offset, (const int64_t *)ctx->ev_start.p,
        (const int64_t *)ctx->ev_len.p, (const int *)ctx->seg_event.p, (const int64_t *)ctx->seg_start.p,
        (const int64_t *)ctx->seg_end.p, (const double *)ctx->seg_mean.p, (const double *)ctx->seg_std.p,
        (const double *)ctx->seg_min.p, (const double *)ctx->seg_max.p, (long long *)dev_out);
    LAUNCHED(ctx);
    return PP_OK;
}

// ---- control exchange over peer memory -------------------------------------------------------------------------
int pp_ctl_create(pp_ctx *ctx, int rank, int world, void *ipc_handle_out, void **local_ptr_out)
{
    if (!ctx || rank < 0 || world < 1 || world > PP_MAX_WORLD || rank >= world)
        return fail(ctx, PP_ERR_ARG, "bad control-exchange arguments");
    CKR(set_device(ctx));
    const size_t bytes = sizeof(unsigned long long) * 2 * (size_t)world * PP_CTL_SLOT;
    CKR(ensure(ctx, ctx->ctl_buf, bytes));
    CK(cudaMemsetAsync(ctx->ctl_buf.p, 0, ctx->ctl_buf.cap, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->ctl_rank = rank;
    ctx->ctl_world = world;
    ctx->ctl_seq = 0;
    if (ipc_handle_out) {
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, ctx->ctl_buf.p));
        memcpy(ipc_handle_out, &h, sizeof h);
    }
    if (local_ptr_out) *local_ptr_out = ctx->ctl_buf.p;
    return PP_OK;
}

int pp_ctl_open(pp_ctx *ctx, const void *ipc_handles, void *const *local_ptrs)
{
    if (!ctx || ctx->ctl_world < 1 || (!ipc_handles && !local_ptrs))
        return fail(ctx, PP_ERR_ARG, "pp_ctl_create first; handles or pointers of every rank");
    CKR(set_device(ctx));
    for (int q = 0; q < ctx->ctl_world; ++q) {
        if (q == ctx->ctl_rank) { ctx->ctl_peers[q] = ctx->ctl_buf.p; continue; }
        if (local_ptrs) { ctx->ctl_peers[q] = local_ptrs[q]; continue; }   // same process: the pointer itself
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)ipc_handles + (size_t)q * sizeof h, sizeof h);
        CK(cudaIpcOpenMemHandle(&ctx->ctl_peers[q], h, cudaIpcMemLazyEnablePeerAccess));
        ctx->ctl_ipc[q] = true;
    }
    CKR(ensure(ctx, ctx->ctl_peers_dev, sizeof(void *) * PP_MAX_WORLD));
    CK(cudaMemcpyAsync(ctx->ctl_peers_dev.p, ctx->ctl_peers, sizeof(void *) * (size_t)ctx->ctl_world,
                       cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

int pp_ctl_exchange(pp_ctx *ctx, const void *dev_src, int n_words, void *dev_dst)
{
    if (!ctx || !dev_src || !dev_dst || n_words < 1 || n_words > PP_CTL_PAYLOAD)
        return fail(ctx, PP_ERR_ARG, "bad control record");
    if (!ctx->ctl_peers_dev.p) return fail(ctx, PP_ERR_STATE, "pp_ctl_open has not run");
    CKR(set_device(ctx));
    const unsigned long long seq = ++ctx->ctl_seq;
    k_ctl_exchange<<<1, 64, 0, ctx->stream>>>((unsigned long long *const *)ctx->ctl_peers_dev.p, ctx->ctl_rank,
                                              ctx->ctl_world, seq, (const unsigned long long *)dev_src, n_words,
                                              (unsigned long long *)dev_dst, ctx->ctr);
    LAUNCHED(ctx);
    return PP_OK;
}

int pp_unpack_tables(pp_ctx *ctx, const int64_t *dev_gathered, int world, int64_t words_per_rank,
                     const int64_t *dev_records, const pp_unpacked_tables *out, int out_is_host, void *cuda_stream)
{
    return pp_unpack_tables_range(ctx, dev_gathered, world, words_per_rank, dev_records, 0, world, out, out_is_host,
                                  cuda_stream);
}

int pp_unpack_tables_range(pp_ctx *ctx, const int64_t *dev_gathered, int world, int64_t words_per_rank,
                           const int64_t *dev_records, int rank_lo, int rank_hi, const pp_unpacked_tables *out,
                           int out_is_host, void *cuda_stream)
{
    if (!ctx || !dev_gathered || !dev_records || !out || world < 1 || world > PP_MAX_WORLD || words_per_rank < 0 ||
        rank_lo < 0 || rank_hi > world || rank_lo >= rank_hi ||
        (words_per_rank & 1) || !out->ev_start || !out->ev_len || !out->seg_event || !out->seg_start ||
        !out->seg_end || !out->mean || !out->std || !out->min || !out->max)
        return fail(ctx, PP_ERR_ARG, "bad unpack arguments");
    CKR(set_device(ctx));
    PPUnpacked O;
    O.cap_events = out->cap_events;
    O.cap_segments = out->cap_segments;
    void *src[9] = {out->ev_start, out->ev_len, out->seg_event, out->seg_start, out->seg_end,
                    out->mean, out->std, out->min, out->max};
    void *dst[9];
    for (int i = 0; i < 9; ++i) {
        dst[i] = src[i];
        // device-visible aliases of page-locked buffers (pp_host_alloc); fails for pageable memory
        if (out_is_host) CK(cudaHostGetDevicePointer(&dst[i], src[i], 0));
    }
    O.ev_start = (long long *)dst[0]; O.ev_len = (long long *)dst[1];
    O.seg_event = (long long *)dst[2]; O.seg_start = (long long *)dst[3]; O.seg_end = (long long *)dst[4];
    O.mean = (double *)dst[5]; O.sd = (double *)dst[6]; O.mn = (double *)dst[7]; O.mx = (double *)dst[8];
    CKR(ensure(ctx, ctx->unpack_flag, 256));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    CK(cudaMemsetAsync(ctx->unpack_flag.p, 0, sizeof(unsigned), st));
    k_unpack_tables<<<ctx->sm_count * 4, 256, 0, st>>>(
        (const long long *)dev_gathered, world, words_per_rank, (const long long *)dev_records, rank_lo, rank_hi, O,
        (unsigned *)ctx->unpack_flag.p);
    LAUNCHED(ctx);
    if (cuda_stream) return PP_OK;   // the caller synchronises with its stream (and sized the tables from the counts)
    unsigned flag = 0;
    CK(cudaMemcpyAsync(&flag, ctx->unpack_flag.p, sizeof flag, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));   // the rows are in the caller's memory when this returns
    if (flag & 1u) return fail(ctx, PP_ERR_CAPACITY, "unpack tables too small");
    if (flag & 2u) return fail(ctx, PP_ERR_CAPACITY, "a rank's packed tables are longer than words_per_rank");
    return PP_OK;
}

// Same pipeline fed from host memory: the trace is copied in chunks on a second stream and every
// stage up to the split search runs on the events completed so far while the next chunk is in flight.
// With host tables (pp_pipeline_host_tables) compaction, statistics and the copy-out of the finished rows also
// run per chunk, so that only the last chunk's rows are left when the last copy has landed.
// `kind`: PP_SRC_TRACE32 (float32 samples) or PP_SRC_ADC16 (int16 counts decoded with `adc`).
static int pipeline_host_impl(pp_ctx *ctx, const void *host, int kind, PPAdc adc, int64_t n, int64_t chunk_samples,
                              const pp_pipeline_params *p, const pp_host_tables *tables, int64_t out[4])
{
    if (!ctx || !p || !host || n <= 0) return fail(ctx, PP_ERR_ARG, "bad trace");
    const size_t elem = sample_bytes(kind);
    CKR(set_device(ctx));
    PPHostTables H;
    memset(&H, 0, sizeof H);
    if (tables) {
        if (tables->cap_events < 0 || tables->cap_segments < 0 || !tables->ev_start || !tables->ev_len ||
            !tables->seg_event || !tables->seg_start || !tables->seg_end ||
            (p->with_stats && (!tables->mean || !tables->std || !tables->min || !tables->max)))
            return fail(ctx, PP_ERR_ARG, "incomplete host tables");
        H.cap_events = tables->cap_events;
        H.cap_segments = tables->cap_segments;
        // device-visible aliases of the page-locked buffers (pp_host_alloc); fails for pageable memory
        CK(cudaHostGetDevicePointer((void **)&H.ev_start, tables->ev_start, 0));
        CK(cudaHostGetDevicePointer((void **)&H.ev_len, tables->ev_len, 0));
        CK(cudaHostGetDevicePointer((void **)&H.seg_event, tables->seg_event, 0));
        CK(cudaHostGetDevicePointer((void **)&H.seg_start, tables->seg_start, 0));
        CK(cudaHostGetDevicePointer((void **)&H.seg_end, tables->seg_end, 0));
        if (p->with_stats) {
            CK(cudaHostGetDevicePointer((void **)&H.mean, tables->mean, 0));
            CK(cudaHostGetDevicePointer((void **)&H.sd, tables->std, 0));
            CK(cudaHostGetDevicePointer((void **)&H.mn, tables->min, 0));
            CK(cudaHostGetDevicePointer((void **)&H.mx, tables->max, 0));
        }
    }
    // 16 Mi samples measured best on B200 (scripts/e2e_breakdown.py: 1 Mi 17.9 ms, 4 Mi 5.9, 8 Mi 5.15, 16 Mi
    // 4.92 for a 60 M-sample trace whose bare copy takes 4.32 ms; a shrinking schedule 24 -> 4 Mi was slower:
    // every chunk pays a full split-search latency)
    if (chunk_samples <= 0) chunk_samples = (int64_t)16 << 20;
    chunk_samples = (chunk_samples + K1_TILE - 1) / K1_TILE * K1_TILE;
    // the whole resident trace in one pass, then its rows to the host tables
    auto whole = [&]() -> int {
        CKR(pp_pipeline(ctx, p, out));
        return tables ? export_tables(ctx, H, p->with_stats) : PP_OK;
    };
    if (p->filter_ncoef > 0 || n <= chunk_samples) {
        // filtering needs every event before the split; a short trace gains nothing from chunking
        if (kind == PP_SRC_ADC16) CKR(pp_trace_upload_adc16(ctx, (const int16_t *)host, n, adc.scale, adc.offset));
        else CKR(pp_trace_upload(ctx, (const float *)host, n, 0));
        return whole();
    }
    CKR(ensure_copy_stream(ctx));
    CKR(ensure(ctx, ctx->trace_buf, elem * (size_t)n));
    set_trace(ctx, ctx->trace_buf.p, kind, n, (int64_t)(ctx->trace_buf.cap / elem));
    ctx->adc = adc;
    ctx->src_kind = kind;
    ctx->flat_cap = n;
    reset_stages(ctx);
    CKR(begin_threshold(ctx, n));
    CKR(prepare_split(ctx, p->min_width, p->max_width, p->window_width));
    // the copies must not overtake earlier work that still reads the trace buffer
    CK(cudaEventRecord(ctx->compute_ev, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->compute_ev, 0));
    for (int64_t a = 0; a < n; a += chunk_samples) {
        const int64_t b = a + chunk_samples < n ? a + chunk_samples : n;
        CK(cudaMemcpyAsync((char *)ctx->trace_buf.p + elem * a, (const char *)host + elem * a, elem * (size_t)(b - a),
                           cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(ctx->copy_ev, ctx->copy_stream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->copy_ev, 0));
        CKR(enqueue_threshold_tiles(ctx, p->threshold, b, (b - a + K1_TILE - 1) / K1_TILE));
        CKR(enqueue_select(ctx, p->rule_mask, p->duration_gt, p->duration_lt, p->min_gt, p->max_lt, 0, 0,
                           b == n ? 2 : 1));
        CKR(enqueue_prefix(ctx, p->prefix_mode));
        CKR(enqueue_search(ctx, p->min_width, p->max_width, p->window_width, p->min_gain));
        if (tables) {  // the events of this chunk are final: their rows leave for the host now
            CKR(enqueue_compact(ctx));
            if (p->with_stats) CKR(enqueue_stats(ctx));
            CKR(enqueue_export(ctx, H, p->with_stats));
        }
    }
    if (!tables) {
        CKR(enqueue_compact(ctx));
        if (p->with_stats) CKR(enqueue_stats(ctx));
    }
    CKR(fetch_counters(ctx));
    const int64_t runs = (int64_t)ctx->h_ctr->n_runs;
    if (runs > ctx->cap_runs) {  // rare: noisy trace with many crossings; the trace is resident now, redo it whole
        CKR(ensure_run_buffers(ctx, runs + 16));
        return whole();
    }
    ctx->n_runs = runs;
    ctx->prefix_valid = true;
    CKR(commit_counters(ctx, out));
    ctx->stats_valid = p->with_stats != 0;
    if (ctx->h_ctr->overflow & PP_OVF_EXPORT) return fail(ctx, PP_ERR_CAPACITY, "host tables too small");
    return PP_OK;
}

static const PPAdc PP_NO_ADC = {1.0, 0.0};

int pp_pipeline_host(pp_ctx *ctx, const float *host, int64_t n, int64_t chunk_samples,
                     const pp_pipeline_params *p, int64_t out[4])
{
    return pipeline_host_impl(ctx, host, PP_SRC_TRACE32, PP_NO_ADC, n, chunk_samples, p, nullptr, out);
}

int pp_pipeline_host_tables(pp_ctx *ctx, const float *host, int64_t n, int64_t chunk_samples,
                            const pp_pipeline_params *p, const pp_host_tables *tables, int64_t out[4])
{
    if (!tables) return fail(ctx, PP_ERR_ARG, "no host tables");
    return pipeline_host_impl(ctx, host, PP_SRC_TRACE32, PP_NO_ADC, n, chunk_samples, p, tables, out);
}

int pp_pipeline_host_adc16(pp_ctx *ctx, const int16_t *host, int64_t n, double scale, double offset,
                           int64_t chunk_samples, const pp_pipeline_params *p, const pp_host_tables *tables,
                           int64_t out[4])
{
    if (pp_adc16_check(scale, offset) != PP_OK)
        return fail(ctx, PP_ERR_ARG, "ADC scale must be finite and non-zero, offset finite, every count decoding finite");
    return pipeline_host_impl(ctx, host, PP_SRC_ADC16, PPAdc{scale, offset}, n, chunk_samples, p, tables, out);
}

// ---- HMM decoding (csrc/hmm.cuh) -----------------------------------------------
// The model as the block of doubles the kernels stage in shared memory; PP_ERR_ARG for S outside 1..128
static int hmm_upload_model(pp_ctx *ctx, const pp_hmm *m)
{
    if (!m) return fail(ctx, PP_ERR_ARG, "no model");
    const int S = m->n_states;
    if (S < 1 || S > HMM_MAX_STATES) return fail(ctx, PP_ERR_ARG, "n_states must be 1..%d, got %d", HMM_MAX_STATES, S);
    if (!m->mean || !m->inv_std || !m->log_norm || !m->log_start || !m->log_trans)
        return fail(ctx, PP_ERR_ARG, "incomplete model");
    const size_t W = hmm_model_words(S);
    std::vector<double> blk;
    CKR(host_scratch(ctx, blk, W));
    for (int j = 0; j < S; ++j) {
        blk[j] = m->mean[j];
        blk[S + j] = m->inv_std[j];
        blk[2 * S + j] = m->log_norm[j];
        blk[3 * S + j] = m->log_start[j];
        blk[4 * S + j] = m->log_end ? m->log_end[j] : 0.0;
    }
    memcpy(blk.data() + 5 * S, m->log_trans, sizeof(double) * (size_t)S * S);
    CKR(ensure(ctx, ctx->hmm_model, sizeof(double) * W));
    CK(cudaMemcpyAsync(ctx->hmm_model.p, blk.data(), sizeof(double) * W, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));   // pageable block: consumed before it is freed
    return PP_OK;
}

static int hmm_grid(pp_ctx *ctx, const void *kernel, int threads, size_t smem, int64_t want, int *grid)
{
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    int64_t g = (int64_t)ctx->sm_count * (per_sm > 0 ? per_sm : 1);
    *grid = (int)(g < want ? g : want);
    return PP_OK;
}

// Decode the sequences x[off[k] .. off[k+1]) (device memory, n_seq of them over n_rows samples) with the staged model
static int hmm_enqueue_decode(pp_ctx *ctx, int S, int algorithm, const double *x, const int64_t *off, int64_t n_seq,
                              int64_t n_rows)
{
    const bool vit = algorithm == 0;
    CKR(ensure(ctx, ctx->hmm_logp, sizeof(double) * (size_t)(n_seq > 0 ? n_seq : 1)));
    CKR(ensure(ctx, ctx->hmm_next, sizeof(unsigned long long)));
    if (vit) {
        CKR(ensure(ctx, ctx->hmm_state, sizeof(int) * (size_t)(n_rows > 0 ? n_rows : 1)));
        CKR(ensure(ctx, ctx->hmm_bp, (size_t)(n_rows > 0 ? n_rows : 1) * S));
    }
    ctx->hmm_n_seq = n_seq;
    ctx->hmm_n_rows = n_rows;
    ctx->hmm_states = vit;
    if (n_seq == 0) return PP_OK;
    HMMSeqs Q;
    Q.x = x;
    Q.off = off;
    Q.n = n_seq;
    Q.logp = (double *)ctx->hmm_logp.p;
    Q.state = vit ? (int *)ctx->hmm_state.p : nullptr;
    Q.bp = vit ? (unsigned char *)ctx->hmm_bp.p : nullptr;
    Q.next = (unsigned long long *)ctx->hmm_next.p;
    CK(cudaMemsetAsync(Q.next, 0, sizeof(unsigned long long), ctx->stream));
    const size_t model_bytes = sizeof(double) * hmm_model_words(S);
    const double *model = (const double *)ctx->hmm_model.p;
    int grid = 0;
    if (S <= 32) {
        const int64_t want = (n_seq + HMM_WARP_THREADS / 32 - 1) / (HMM_WARP_THREADS / 32);
        if (vit) {
            CKR(hmm_grid(ctx, (const void *)k_hmm_warp<true>, HMM_WARP_THREADS, model_bytes, want, &grid));
            k_hmm_warp<true><<<grid, HMM_WARP_THREADS, model_bytes, ctx->stream>>>(model, S, Q);
        } else {
            CKR(hmm_grid(ctx, (const void *)k_hmm_warp<false>, HMM_WARP_THREADS, model_bytes, want, &grid));
            k_hmm_warp<false><<<grid, HMM_WARP_THREADS, model_bytes, ctx->stream>>>(model, S, Q);
        }
    } else {
        const size_t smem = model_bytes + sizeof(double) * 2 * HMM_MAX_STATES;
        if (vit) {
            CKR(hmm_grid(ctx, (const void *)k_hmm_cta<true>, HMM_CTA_THREADS, smem, n_seq, &grid));
            k_hmm_cta<true><<<grid, HMM_CTA_THREADS, smem, ctx->stream>>>(model, S, Q);
        } else {
            CKR(hmm_grid(ctx, (const void *)k_hmm_cta<false>, HMM_CTA_THREADS, smem, n_seq, &grid));
            k_hmm_cta<false><<<grid, HMM_CTA_THREADS, smem, ctx->stream>>>(model, S, Q);
        }
    }
    LAUNCHED(ctx);
    if (vit) {
        const int64_t tb = (n_seq + 127) / 128;
        k_hmm_traceback<<<(unsigned)(tb < ctx->sm_count * 8 ? tb : ctx->sm_count * 8), 128, 0, ctx->stream>>>(Q, S);
        LAUNCHED(ctx);
    }
    return PP_OK;
}

// Merge runs of segments that share a Viterbi state: new breakpoints, the existing compaction and K4 statistics
static int hmm_enqueue_merge(pp_ctx *ctx)
{
    const int64_t n_old = ctx->n_segments;
    const unsigned grid = (unsigned)ctx->sm_count * 4;
    CKR(ensure(ctx, ctx->hmm_old_flat, sizeof(int64_t) * (size_t)(n_old > 0 ? n_old : 1)));
    CKR(ensure(ctx, ctx->hmm_old_state, sizeof(int) * (size_t)(n_old > 0 ? n_old : 1)));
    if (n_old > 0) {
        CK(cudaMemcpyAsync(ctx->hmm_old_flat.p, ctx->seg_flat.p, sizeof(int64_t) * n_old, cudaMemcpyDeviceToDevice,
                           ctx->stream));
        CK(cudaMemcpyAsync(ctx->hmm_old_state.p, ctx->hmm_state.p, sizeof(int) * n_old, cudaMemcpyDeviceToDevice,
                           ctx->stream));
    }
    CK(cudaMemsetAsync(ctx->bits.p, 0, sizeof(unsigned) * ctx->n_words, ctx->stream));
    k_hmm_merge_bits<<<grid, 256, 0, ctx->stream>>>((const int *)ctx->seg_event.p, (const int64_t *)ctx->seg_flat.p,
                                                    (const int *)ctx->hmm_state.p, n_old, (unsigned *)ctx->bits.p);
    LAUNCHED(ctx);
    // the whole table is rebuilt: no range was finalised (the streamed export leaves these at the totals)
    CK(cudaMemsetAsync(&ctx->ctr->seg_done, 0, 3 * sizeof(unsigned long long), ctx->stream));
    CKR(enqueue_compact(ctx));
    k_hmm_merged_states<<<grid, 256, 0, ctx->stream>>>(ctx->ctr, (const int64_t *)ctx->seg_flat.p,
                                                       (const int64_t *)ctx->hmm_old_flat.p,
                                                       (const int *)ctx->hmm_old_state.p, n_old, (int *)ctx->hmm_state.p);
    LAUNCHED(ctx);
    CKR(launch_stats(ctx, 0, (const int64_t *)ctx->seg_flat.p, (const int *)ctx->seg_event.p, ctx->cap_segs,
                     (double *)ctx->seg_mean.p, (double *)ctx->seg_std.p, (double *)ctx->seg_min.p,
                     (double *)ctx->seg_max.p));
    CKR(fetch_counters(ctx));
    CKR(check_overflow(ctx));
    ctx->n_segments = (int64_t)ctx->h_ctr->n_segments;
    ctx->hmm_n_rows = ctx->n_segments;
    return PP_OK;
}

int pp_hmm_decode(pp_ctx *ctx, const pp_hmm *model, int algorithm, int merge, int64_t *n_segments)
{
    if (!ctx) return PP_ERR_ARG;
    if (algorithm != 0 && algorithm != 1) return fail(ctx, PP_ERR_ARG, "algorithm must be 0 (Viterbi) or 1 (forward)");
    if (merge && algorithm != 0) return fail(ctx, PP_ERR_ARG, "merging needs Viterbi states");
    if (!model || model->n_states < 1 || model->n_states > HMM_MAX_STATES)
        return fail(ctx, PP_ERR_ARG, "n_states must be 1..%d", HMM_MAX_STATES);
    if (ctx->n_segments < 0 || !ctx->stats_valid || ctx->n_events < 0)
        return fail(ctx, PP_ERR_STATE, "no resident segment statistics (pp_statsplit + pp_segment_stats / pp_pipeline)");
    CKR(set_device(ctx));
    CKR(hmm_upload_model(ctx, model));
    const int64_t E = ctx->n_events, R = ctx->n_segments;
    CKR(ensure(ctx, ctx->hmm_off, sizeof(int64_t) * (size_t)(E + 1)));
    k_hmm_event_offsets<<<(unsigned)(E / 256 + 1 < ctx->sm_count * 4 ? E / 256 + 1 : ctx->sm_count * 4), 256, 0,
                          ctx->stream>>>((const int *)ctx->seg_event.p, R, E, (int64_t *)ctx->hmm_off.p);
    LAUNCHED(ctx);
    CKR(hmm_enqueue_decode(ctx, model->n_states, algorithm, (const double *)ctx->seg_mean.p,
                           (const int64_t *)ctx->hmm_off.p, E, R));
    if (merge) CKR(hmm_enqueue_merge(ctx));
    if (n_segments) *n_segments = ctx->n_segments;
    return PP_OK;
}

int pp_hmm_decode_sequences(pp_ctx *ctx, const pp_hmm *model, int algorithm, const double *x, const int64_t *len,
                            int64_t n)
{
    if (!ctx) return PP_ERR_ARG;
    if (algorithm != 0 && algorithm != 1) return fail(ctx, PP_ERR_ARG, "algorithm must be 0 (Viterbi) or 1 (forward)");
    if (n < 0 || (n > 0 && (!x || !len))) return fail(ctx, PP_ERR_ARG, "bad sequences");
    std::vector<int64_t> off;
    CKR(host_scratch(ctx, off, (size_t)(n + 1)));
    off[0] = 0;
    for (int64_t k = 0; k < n; ++k) {
        if (len[k] <= 0) return fail(ctx, PP_ERR_ARG, "sequence %lld is empty", (long long)k);
        off[k + 1] = off[k] + len[k];
    }
    const int64_t total = off[n];
    CKR(set_device(ctx));
    CKR(hmm_upload_model(ctx, model));
    CKR(ensure(ctx, ctx->hmm_off, sizeof(int64_t) * (size_t)(n + 1)));
    CKR(ensure(ctx, ctx->hmm_x, sizeof(double) * (size_t)(total > 0 ? total : 1)));
    CK(cudaMemcpyAsync(ctx->hmm_off.p, off.data(), sizeof(int64_t) * (size_t)(n + 1), cudaMemcpyHostToDevice,
                       ctx->stream));
    if (total) CK(cudaMemcpyAsync(ctx->hmm_x.p, x, sizeof(double) * (size_t)total, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));   // pageable host memory: consumed before the call returns
    return hmm_enqueue_decode(ctx, model->n_states, algorithm, (const double *)ctx->hmm_x.p,
                              (const int64_t *)ctx->hmm_off.p, n, total);
}

int pp_hmm_download(pp_ctx *ctx, int64_t cap_seq, double *log_prob, int64_t cap_states, int32_t *state)
{
    if (!ctx) return PP_ERR_ARG;
    if (ctx->hmm_n_seq < 0) return fail(ctx, PP_ERR_STATE, "no HMM decode has run");
    if (state && !ctx->hmm_states) return fail(ctx, PP_ERR_STATE, "the last decode computed no states (forward)");
    if ((log_prob && cap_seq < ctx->hmm_n_seq) || (state && cap_states < ctx->hmm_n_rows))
        return fail(ctx, PP_ERR_CAPACITY, "HMM result buffers too small");
    CKR(set_device(ctx));
    if (log_prob && ctx->hmm_n_seq)
        CK(cudaMemcpyAsync(log_prob, ctx->hmm_logp.p, sizeof(double) * (size_t)ctx->hmm_n_seq, cudaMemcpyDeviceToHost,
                           ctx->stream));
    if (state && ctx->hmm_n_rows)
        CK(cudaMemcpyAsync(state, ctx->hmm_state.p, sizeof(int) * (size_t)ctx->hmm_n_rows, cudaMemcpyDeviceToHost,
                           ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PP_OK;
}

}  // extern "C"
