/*
 * pypore_b200.h -- C ABI of libpypore_b200.so: the B200 (sm_100a) implementation
 * of PyPore's signal-segmentation hot path.
 *
 * The reference (jmschrei/PyPore) has no FFI: its plug-in boundary is the
 * duck-typed Python protocol `parser.parse(current) -> [Segment]`
 * (PyPore/parsers.py:57-59) called from File.parse (PyPore/DataTypes.py:589-602),
 * Event.parse (DataTypes.py:276-289) and Event.filter (DataTypes.py:258-274).
 * Each entry point below names the reference lines whose arithmetic it
 * replaces; pypore_b200/ binds them with ctypes (see INTEGRATION.md for the
 * stub a reference maintainer would add).
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success or
 * a negative pp_status, with a message available from pp_last_error(); all work
 * is ordered on the context's CUDA stream; calls that hand data back to the
 * host synchronise that stream before returning.  A context is bound to one
 * device and must not be used from two threads at once (the reference is
 * single-threaded, SURVEY 8b "Threading").
 *
 * Index conventions: trace positions and event starts are int64 sample indices
 * into the trace; segment starts/ends are int64 sample indices RELATIVE to their
 * event (what FastStatSplit.parse returns, cparsers.pyx:115-116).
 */
#ifndef PYPORE_B200_H
#define PYPORE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pp_ctx pp_ctx;

enum pp_status {
    PP_OK = 0,
    PP_ERR_CUDA = -1,      /* a CUDA runtime call failed (message has the cudaError string) */
    PP_ERR_ARG = -2,       /* invalid argument / call order */
    PP_ERR_CAPACITY = -3,  /* a caller-supplied output buffer is too small */
    PP_ERR_STATE = -4,     /* required earlier stage has not run */
    PP_ERR_FILTER_LEN = -5 /* an event is not longer than filtfilt's padlen (scipy raises ValueError) */
};

/* Rule mask for pp_select_events: the three default-shaped rules of
 * lambda_event_parser (parsers.py:133-135). */
enum pp_rule {
    PP_RULE_DURATION_GT = 1, /* event.duration > duration_gt  (samples) */
    PP_RULE_MIN_GT = 2,      /* event.min > min_gt */
    PP_RULE_MAX_LT = 4,      /* event.max < max_lt */
    PP_RULE_DURATION_LT = 8  /* event.duration < duration_lt (GUI rule, parsers.py:207) */
};

/* Prefix-sum strategy for FastStatSplit's cumsums (cparsers.pyx:110-111). */
enum pp_prefix_mode {
    PP_PREFIX_AUTO = 0,       /* parallel scan with exactness check, sequential redo of inexact events */
    PP_PREFIX_SEQUENTIAL = 1, /* strict np.cumsum order, one thread per event */
    PP_PREFIX_PARALLEL = 2    /* parallel scan only (bit-identical iff all sums are exact) */
};

/* ---- context ---------------------------------------------------------- */
int pp_version(void);
int pp_device_count(void);
/* stream == NULL: the context creates its own non-blocking stream. */
int pp_create(int device, void *cuda_stream, pp_ctx **out);
void pp_destroy(pp_ctx *ctx);
const char *pp_last_error(pp_ctx *ctx);
int pp_sync(pp_ctx *ctx);
/* The CUDA stream (cudaStream_t) all of the context's work is ordered on. */
void *pp_stream(pp_ctx *ctx);
/* Page-locked host memory (cudaMallocHost) for traces handed to pp_pipeline_host /
 * pp_trace_upload and for table downloads: copies to and from it run at full PCIe rate. */
int pp_host_alloc(pp_ctx *ctx, int64_t bytes, void **out);
void pp_host_free(pp_ctx *ctx, void *p);
/* Options: PP_OPT_SCREEN (default 1) -- 1: two-stage split search (bounded-error
 * screening of every candidate, exact arithmetic for the contenders); 0: exact
 * arithmetic for every candidate (validation mode, same results, many times slower). */
enum pp_option {
    PP_OPT_SCREEN = 0,
    /* PP_OPT_SPINE (default 1) -- 1: events longer than the locally resolvable interval are first walked window by
     * window by a thread-block cluster each (k3_spine: 4 CTAs x 512 threads, summaries through distributed shared
     * memory); 0: the 128-thread work-queue CTAs walk them (same results). */
    PP_OPT_SPINE = 1,
    /* PP_OPT_SPLIT_CTAS (default 0) -- number of persistent CTAs the split search (k3_split) is launched with; 0 or
     * anything above one full wave: one full wave (7 CTAs per SM).  The search is a work queue, any CTA count gives the
     * same tables.  Contexts that share a GPU (pypore_b200/batch.py: several files in flight, each with a few
     * hundred events) take a fraction of a wave each, so that their searches are resident side by side instead of
     * one after the other. */
    PP_OPT_SPLIT_CTAS = 2,
    /* PP_OPT_SPLIT_KERNEL -- which kernel runs the split search: 0: k3_split, CTAs that resolve a task level by level
     * between barriers; 1: k3_flow, every warp an independent worker on a CTA-shared stack of window pieces, no
     * barriers.  Same tables bit for bit (the result of a window depends only on its interval and the prefix sums). */
    PP_OPT_SPLIT_KERNEL = 3
};
int pp_set_option(pp_ctx *ctx, int option, int64_t value);
/* The current value of an option (so that a caller can restore it). */
int pp_get_option(pp_ctx *ctx, int option, int64_t *value);
/* Number of kernel launches this context has issued since creation. */
int64_t pp_launch_count(pp_ctx *ctx);
/* Milliseconds between two internal CUDA events bracketing the named stage of
 * the LAST pipeline call: 0 threshold, 1 select, 2 filter, 3 prefix, 4 split,
 * 5 compact, 6 stats.  Valid after pp_sync(). */
int pp_stage_ms(pp_ctx *ctx, int stage, float *ms);

/* ---- trace residency -------------------------------------------------- */
/* Copy a host float32 trace to the device (replaces File.current,
 * DataTypes.py:572-583).  `extra_capacity` samples are reserved after the trace
 * for pp_trace_append (multi-GPU halo). */
int pp_trace_upload(pp_ctx *ctx, const float *host, int64_t n, int64_t extra_capacity);
/* Same for a float64 trace -- what the reference's own loader produces (PyPore/read_abf.py:208-210: int16 ADC counts
 * times a float64 scale factor).  The trace stays float64 on the device (8 B per sample): the threshold scan
 * compares the doubles themselves, run extrema are the doubles' own, and the later stages read the events out of
 * it like out of a float32 trace.  pp_trace_append / pp_trace_extend are float32-only, and the streamed host pipeline
 * takes float32 or int16 ADC input. */
int pp_trace_upload_f64(pp_ctx *ctx, const double *host, int64_t n);
/* Same for int16 ADC counts, 2 B per sample over the link and in the scan: every stage behaves as if it had been
 * handed the float64 trace decode(c) = fl(fl(c * scale) + offset) (two roundings, no FMA: what NumPy computes for
 * counts.astype(np.float64) * scale + offset).  The threshold scan compares integer keys (pp_adc16_key_threshold),
 * the run extrema are decoded from the extreme keys, the later stages decode samples where they read them.
 * PP_ERR_ARG unless scale is finite and non-zero, offset finite and every count decodes to a finite value.
 * pp_trace_append / extend / prefetch / adopt and the pp_shard_* calls are float32-only: PP_ERR_STATE while an ADC
 * trace is resident. */
int pp_trace_upload_adc16(pp_ctx *ctx, const int16_t *host, int64_t n, double scale, double offset);
/* PP_OK if (scale, offset) is a valid ADC decoding (see above), PP_ERR_ARG otherwise.  No context, no device. */
int pp_adc16_check(double scale, double offset);
/* The threshold scan's view of `current < threshold` for ADC counts: with kxor = -1 for a negative scale and 0
 * otherwise, the decoded current is non-decreasing in the key k = c ^ kxor, and decode(c) < threshold holds exactly
 * when k < *key (*key = 32768: for every count; -32768: for none, a NaN threshold included).  No context, no
 * device; PP_ERR_ARG for an invalid decoding. */
int pp_adc16_key_threshold(double scale, double offset, double threshold, int32_t *key, int32_t *kxor);
/* Back-to-back traces: pp_trace_prefetch starts the copy of the NEXT float32 trace (ideally from page-locked memory)
 * into another device buffer on the context's copy stream and returns at once -- it runs under whatever the
 * context's stream is doing with the current trace; pp_trace_swap makes the oldest prefetched trace the resident one
 * (the context's stream waits for its copy, the host does not).  Up to TWO traces may be waiting for their swap
 * (PP_ERR_STATE beyond that): with two, the copy stream always has the next copy queued behind the running one and
 * the upload link never idles between steps.  Three trace buffers live at most. */
int pp_trace_prefetch(pp_ctx *ctx, const float *host, int64_t n, int64_t extra_capacity);
int pp_trace_swap(pp_ctx *ctx);
/* Duration in milliseconds of the copy that brought up the trace pp_trace_swap made resident last (waits for it).  A caller that
 * shards one trace over the GPUs of a node uses it to cut the trace in proportion to what each GPU's upload path
 * delivers when all of them copy at once. */
int pp_trace_prefetch_ms(pp_ctx *ctx, float *ms);
/* Use device memory the caller owns (no copy; must stay valid; capacity in samples). */
int pp_trace_adopt(pp_ctx *ctx, const float *dev, int64_t n, int64_t capacity);
/* Append `n` samples (device or host pointer) after the current trace end: the
 * continuation of an event that straddles this GPU's chunk boundary. */
int pp_trace_append(pp_ctx *ctx, const float *src, int64_t n, int src_is_device);
/* Drop samples appended after position `n` (start of a new multi-GPU step). */
int pp_trace_truncate(pp_ctx *ctx, int64_t n);
/* Declare that the caller wrote `n` samples directly after the current trace end (NCCL recv or a
 * peer copy into pp_trace_device_ptr() + pp_trace_len(), within the reserved capacity). */
int pp_trace_extend(pp_ctx *ctx, int64_t n);
int64_t pp_trace_len(pp_ctx *ctx);
const float *pp_trace_device_ptr(pp_ctx *ctx);

/* ---- K1: lambda_event_parser.parse (parsers.py:142-155) -------------- */
/* Runs of consecutive samples on one side of the threshold, compared as
 * double(x) < threshold, with per-run min/max (core.py:215-220).
 * `scan_len` <= trace length restricts the scan to a prefix of the trace
 * (samples appended as halo are not re-scanned); pass -1 for the whole trace. */
int pp_threshold_scan(pp_ctx *ctx, double threshold, int64_t scan_len, int64_t *n_runs);
int pp_runs_download(pp_ctx *ctx, int64_t cap, int64_t *start, int64_t *length, double *mn,
                     double *mx, uint8_t *below);
/* Rows [first, first+count) of the run table (multi-GPU: only the boundary runs travel). */
int pp_runs_download_range(pp_ctx *ctx, int64_t first, int64_t count, int64_t *start, int64_t *length,
                           double *mn, double *mx, uint8_t *below);
/* _lambda_select for default-shaped rules, evaluated on the device
 * (parsers.py:133-140).  Runs flagged in `skip_first`/`skip_last` (0/1) are
 * excluded regardless of the rules (multi-GPU: a run owned by a neighbour). */
int pp_select_events(pp_ctx *ctx, int rule_mask, int64_t duration_gt, int64_t duration_lt,
                     double min_gt, double max_lt, int skip_first, int skip_last,
                     int64_t *n_events, int64_t *n_event_samples);
/* Events chosen by the host (arbitrary Python rules evaluated on the run table). */
int pp_set_events(pp_ctx *ctx, const int64_t *start, const int64_t *length, int64_t n_events);
/* Append one event after the current last event (multi-GPU: the run that starts
 * in this GPU's chunk and continues into the halo appended with pp_trace_append). */
int pp_append_event(pp_ctx *ctx, int64_t start, int64_t length);
int pp_events_download(pp_ctx *ctx, int64_t cap, int64_t *start, int64_t *length);

/* ---- float64 events supplied directly (SpeedyStatSplit.parse(current)) */
/* `n_events` float64 events packed back to back in `host` (lengths in `length`). */
int pp_events_upload_f64(pp_ctx *ctx, const double *host, const int64_t *length, int64_t n_events);

/* ---- K5: Event.filter (DataTypes.py:258-274; scipy.signal.filtfilt) -- */
/* Zero-phase IIR filter of every current event; b, a have `ncoef` entries
 * (a[0] == 1), zi has ncoef-1 (scipy.signal.lfilter_zi).  Afterwards the events'
 * current is the float64 filtered signal (later stages read it). */
int pp_filter_events(pp_ctx *ctx, const double *b, const double *a, const double *zi, int ncoef);
/* Event samples as float64, packed back to back (filtered if a filter ran). */
int pp_event_samples_download(pp_ctx *ctx, int64_t cap, double *out);

/* ---- K2+K3: FastStatSplit.parse (cparsers.pyx:103-203) ---------------- */
/* min_gain is computed by the host exactly as cparsers.pyx:82-101. */
int pp_statsplit(pp_ctx *ctx, int min_width, int max_width, int window_width, double min_gain,
                 int prefix_mode, int64_t *n_segments);
/* Prefix sums only (cparsers.pyx:110-111 / :129-130), for pp_window_gains without a split. */
int pp_prefix(pp_ctx *ctx, int prefix_mode);
/* gain(i) in the reference's exact arithmetic for every candidate of a batch of windows
 * [ps[w], pe[w]) of event `ev`: i = ps+min_width .. pe-min_width (the loop of
 * _best_split_stepwise_score, cparsers.pyx:234-240; with ps=0, pe=len-1, min_width=2 the loop of
 * _best_single_split, cparsers.pyx:142-151).  The gains of window w follow those of window w-1
 * in `out` (host memory, `cap` doubles).  Needs resident prefix sums (pp_prefix / pp_statsplit). */
int pp_window_gains(pp_ctx *ctx, int64_t ev, int n_windows, const int32_t *ps, const int32_t *pe, int min_width,
                    double *out, int64_t cap);

/* ---- K4: Segment.mean/std/min/max (core.py:209-223) ------------------- */
int pp_segment_stats(pp_ctx *ctx);
int pp_segments_download(pp_ctx *ctx, int64_t cap, int32_t *event, int64_t *start, int64_t *end,
                         double *mean, double *std, double *mn, double *mx);
/* Same statistics for the events themselves (Event is a Segment, DataTypes.py:241). */
int pp_event_stats_download(pp_ctx *ctx, int64_t cap, double *mean, double *std, double *mn, double *mx);
/* Device pointers to the compact tables (multi-GPU all-gather reads these):
 * which = 0 seg_event(int32) 1 seg_start(int64) 2 seg_end(int64) 3 mean 4 std 5 min 6 max (f64)
 *         7 ev_start(int64) 8 ev_len(int64). */
const void *pp_table_device_ptr(pp_ctx *ctx, int which);
/* Work counters of the last pp_statsplit: [0] candidate evaluations (same count
 * as the reference's inner loop), [1] window scans, [2] events whose prefix sums
 * were redone sequentially, [3] queue tasks processed, [4] candidates evaluated
 * with the exact reference arithmetic after screening.  How the screened search
 * decided its windows (all 0 with PP_OPT_SCREEN = 0): [5] on the screened gain
 * alone (one contender, clear of min_gain by more than the error bound), [6] by
 * the argmax over the exact gains of several contenders (re-screened pieces
 * included), [7] by an exact scan of every candidate (a candidate failed the
 * validity test, the window cannot be screened, or its exact-evaluation requests
 * overflowed).  Windows with one contender evaluated exactly count in none of
 * [5..7].  The sharded multi-GPU path reports [0], [1] and [4] only. */
int pp_split_counters(pp_ctx *ctx, int64_t out[8]);

/* Validation hook for the screening bound: for window [ps,pe) of event `ev` (prefix sums
 * from the last pp_statsplit), per candidate i = ps+min_width+j: the screened value, the
 * reference-arithmetic value fl(low+high) and the validity flag.  Arrays hold
 * pe-ps-2*min_width+1 entries.  eps receives the bound the kernel applies to this window. */
int pp_debug_screen(pp_ctx *ctx, int64_t ev, int ps, int pe, int min_width, double *h_screen,
                    double *h_exact, uint8_t *ok, double *eps);
/* Validation: the resident prefix sums (K2) of all events, de-interleaved into c (cumsum of x) and c2 (cumsum of
 * x*x), n_event_samples entries each in flat event space, and per event whether the strict-order kernel computed
 * them: the exactness verdict under PP_PREFIX_AUTO, all 0 under PP_PREFIX_PARALLEL, all 1 under
 * PP_PREFIX_SEQUENTIAL.  cap bounds both lengths.  PP_ERR_STATE unless pp_prefix / pp_statsplit ran on the current
 * events. */
int pp_debug_prefix(pp_ctx *ctx, int64_t cap, double *c, double *c2, uint8_t *redone);

/* Validation hook for the hardware term of the screening bound: the largest absolute error,
 * over all 2^23 float32 mantissas in [1, 2), of the 23-bit fixed-point log2 the screening
 * builds from MUFU.LG2 (lg2.approx.f32) and one float32 addition.  The bound in
 * split.cuh assumes <= 2^-22 + 2^-24. */
int pp_debug_lg2_error(pp_ctx *ctx, double *max_err);

/* ---- whole pipeline, no host synchronisation between stages ----------- */
typedef struct pp_pipeline_params {
    double threshold;
    int rule_mask;
    int64_t duration_gt, duration_lt;
    double min_gt, max_lt;
    int filter_ncoef;          /* 0 = no filter */
    const double *filter_b, *filter_a, *filter_zi;
    int min_width, max_width, window_width;
    double min_gain;
    int prefix_mode;
    int with_stats;
} pp_pipeline_params;
/* threshold scan -> select -> [filter] -> prefix -> split -> compact -> stats on
 * the resident trace.  Counts: out[0] runs, out[1] events, out[2] event
 * samples, out[3] segments. */
int pp_pipeline(pp_ctx *ctx, const pp_pipeline_params *p, int64_t out[4]);
/* The same pipeline for a trace in HOST memory (File(current=...).parse(...) end to end): the
 * trace is copied in chunks of `chunk_samples` (<= 0: 16 Mi samples; use pinned memory for an
 * asynchronous copy) on a second stream while the threshold scan, event selection, prefix sums and
 * split search already run on the events completed by the chunks that have arrived; compaction and
 * statistics follow the last chunk.  Results are identical to pp_trace_upload + pp_pipeline.
 * With a filter, or a trace of at most one chunk, it is exactly that sequence. */
int pp_pipeline_host(pp_ctx *ctx, const float *host, int64_t n, int64_t chunk_samples,
                     const pp_pipeline_params *p, int64_t out[4]);
/* pp_pipeline_host that also delivers the event and segment tables to HOST memory: compaction, statistics and
 * the copy-out of the rows a chunk has finalised run per chunk, overlapped with the copy of the next chunk in the
 * other direction, so that only the last chunk's rows are outstanding when the last samples have landed (the
 * rows are written by a kernel straight into the page-locked buffers).  All buffers must come from pp_host_alloc;
 * the statistics columns may be NULL when p->with_stats == 0.  PP_ERR_CAPACITY: the tables were too small --
 * nothing of them is valid, the counts in `out` and the device tables are (download them the usual way). */
typedef struct pp_host_tables {
    int64_t cap_events;
    int64_t *ev_start, *ev_len;
    int64_t cap_segments;
    int32_t *seg_event;
    int64_t *seg_start, *seg_end;
    double *mean, *std, *min, *max;
} pp_host_tables;
int pp_pipeline_host_tables(pp_ctx *ctx, const float *host, int64_t n, int64_t chunk_samples,
                            const pp_pipeline_params *p, const pp_host_tables *tables, int64_t out[4]);
/* pp_pipeline_host / pp_pipeline_host_tables (tables == NULL: device tables only) for int16 ADC counts decoded with
 * `scale` and `offset` (pp_trace_upload_adc16): 2 B per sample over the link, same chunked copy / compute overlap,
 * the same tables the float64 trace decode(counts) gives. */
int pp_pipeline_host_adc16(pp_ctx *ctx, const int16_t *host, int64_t n, double scale, double offset,
                           int64_t chunk_samples, const pp_pipeline_params *p,
                           const pp_host_tables *tables /* NULL: device tables only */, int64_t out[4]);

/* ---- hidden Markov models over segment means (Event.apply_hmm / Event.parse(hmm=), DataTypes.py:292-355) ----
 * S = n_states emitting states (1..128) with normal emissions, every log taken by the host: inv_std[j] = 1/sigma_j,
 * log_norm[j] = -log(sigma_j) - log(2 pi)/2, log_start[j], log_trans[i*S + j] (row-normalised), log_end[j] (NULL:
 * no end term).  Emission e_j(x) = log_norm[j] - 0.5 * z*z, z = (x - mean[j]) * inv_std[j], one rounding per
 * operation and no FMA (bit-equal to NumPy).  algorithm 0: Viterbi -- log-probability of the best path and the path,
 * bit-exact (ties go to the lowest state index); 1: forward log-likelihood (CUDA exp / log, not bit-exact).  A NaN
 * value gives log-probability NaN, an impossible sequence -inf; the states of both are all -1. */
typedef struct pp_hmm {
    int n_states;
    const double *mean, *inv_std, *log_norm, *log_start, *log_trans /* [i*S+j] */, *log_end /* NULL: none */;
} pp_hmm;
/* Decode the resident segment table, one sequence of segment means per event.  merge = 1 (Viterbi only): every run
 * of consecutive segments of one event that share a state >= 0 becomes one segment whose statistics are computed
 * again from the samples (K4, same sample source); *n_segments receives the new row count.  PP_ERR_STATE without
 * resident segment statistics, PP_ERR_ARG for n_states outside 1..128 or merge with forward. */
int pp_hmm_decode(pp_ctx *ctx, const pp_hmm *model, int algorithm, int merge, int64_t *n_segments);
/* Decode n host sequences packed back to back in x (len[k] >= 1 values each). */
int pp_hmm_decode_sequences(pp_ctx *ctx, const pp_hmm *model, int algorithm, const double *x, const int64_t *len,
                            int64_t n);
/* Results of the last decode: one log-probability per sequence, one state per value (per segment row of the
 * merged table after a merge).  state may be NULL; it must be after a forward decode (PP_ERR_STATE otherwise). */
int pp_hmm_download(pp_ctx *ctx, int64_t cap_seq, double *log_prob, int64_t cap_states, int32_t *state);

/* ---- multi-GPU: one context per rank, contiguous trace chunks (SURVEY 8e) -------------
 * The exchange itself (NCCL all-gathers of the records / tables, point-to-point halos) is
 * driven by pypore_b200/dist.py; these calls keep every stage on the device between them.
 * pp_shard_scan: threshold scan of the chunk's first scan_len samples; writes the 12-double
 *   boundary record [n_local, n_runs, first run: below,len,min,max, last run: below,start,len,
 *   min,max, run-table-overflow flag] to DEVICE memory, no host synchronisation.
 * pp_shard_finish: select (first / last run optionally owned by a neighbour), optional
 *   straddling event appended, prefix + split + compaction + statistics; writes the 8-word result
 *   record [runs, events, event samples, segments, overflow flags, candidates, scans, exact
 *   evaluations] to DEVICE memory, no host synchronisation.
 * pp_shard_plan / pp_shard_finish_planned: the same step without the host round trip between scan
 *   and finish.  The caller placed `halo_avail` samples of the right neighbour's chunk after its own
 *   (pp_trace_extend) before anything was known about the runs; pp_shard_plan derives this rank's part of
 *   the boundary plan on the DEVICE from the all-gathered boundary records (world x 12 doubles) and writes
 *   8 words [skip_first, skip_last, has_event, ev_start, ev_len, redo flags, halo samples needed, 0];
 *   pp_shard_finish_planned reads them there.  Word 4 of the result record carries the redo flags
 *   (16: a straddling event needs more than halo_avail samples or spans more than two chunks; 1: a rank's
 *   run table overflowed) -- the caller then repeats the step with pp_shard_finish and a host-made plan.
 * pp_shard_commit: hands the (all-gathered, host-read) result record back so that downloads work.
 * pp_pack_tables: the tables as 8-byte words in one device buffer for ONE all-gather: event rows {global start,
 *   length} (2 words), then segment rows of 4 words {global event id | event-relative start << 32, mean, std,
 *   min | max << 32 as float32 bit patterns} -- 32 B instead of the table's 56: `end` is the next row's start (or
 *   the event's length) and is rebuilt after the gather, and min / max are stored as float32.  That is exact only
 *   when the segment table was computed from a float32 trace's own samples: PP_ERR_STATE otherwise (a float64 or
 *   int16 ADC trace, filtered events, events from pp_events_upload_f64), and nothing is written.  The pp_shard_*
 *   calls themselves take float64 traces too; their tables stay downloadable, only the packing refuses them.
 *   2 E + 4 S words.  Counts and the global event-id base are read on the DEVICE from the all-gathered result
 *   records (8 words per rank), so the call needs no host knowledge of them; nothing is written if cap_words is
 *   too small.
 */
int pp_shard_scan(pp_ctx *ctx, double threshold, int64_t scan_len, double *dev_record);
int pp_shard_finish(pp_ctx *ctx, const pp_pipeline_params *p, int skip_first, int skip_last, int has_event,
                    int64_t ev_start, int64_t ev_len, int64_t *dev_record);
int pp_shard_plan(pp_ctx *ctx, const double *dev_infos, int rank, int world, const pp_pipeline_params *p,
                  int64_t halo_avail, int64_t *dev_plan);
int pp_shard_finish_planned(pp_ctx *ctx, const pp_pipeline_params *p, const int64_t *dev_plan, int64_t *dev_record);
int pp_shard_commit(pp_ctx *ctx, const int64_t rec[8]);
/* pp_ctl_create / pp_ctl_open / pp_ctl_exchange: the control records of a sharded step (12-double boundary record,
 *   8-word result record) without a collective.  pp_ctl_create allocates this rank's record buffer and returns its
 *   CUDA IPC handle (64 bytes; and / or the device pointer, for contexts of ONE process); after the caller has
 *   all-gathered the handles ONCE, pp_ctl_open maps every peer's buffer.  pp_ctl_exchange(src, n_words <= 16, dst)
 *   then enqueues one tiny kernel on the context's stream: it stores this rank's record into every peer's buffer
 *   over NVLink, raises a flag, waits for all ranks' flags in its own buffer and writes the world x n_words gathered
 *   records to dst (device memory) -- what an all-gather of the records would have produced, without NCCL's launch
 *   latency on the step's critical path.  Every rank must call it the same number of times (a sequence number
 *   pairs the calls); a record that does not arrive within seconds raises flag 64 in the result record. */
int pp_ctl_create(pp_ctx *ctx, int rank, int world, void *ipc_handle_out, void **local_ptr_out);
int pp_ctl_open(pp_ctx *ctx, const void *ipc_handles, void *const *local_ptrs);
int pp_ctl_exchange(pp_ctx *ctx, const void *dev_src, int n_words, void *dev_dst);
/* pp_unpack_tables: the all-gathered packed tables (world rows of words_per_rank words -- an even number --, row r
 *   = rank r's pp_pack_tables output) as the caller's tables in one pass, one contiguous array per column:
 *   events {global start, length}, segments {global event id, start, end (int64), mean, std, min, max (float64)};
 *   E / S = the sums over the all-gathered result records (device memory).  out_is_host = 1: the arrays are
 *   page-locked host memory (pp_host_alloc) and are written by the kernel directly -- the call returns when the
 *   rows are there; 0: device memory.  PP_ERR_CAPACITY if cap_events / cap_segments rows do not suffice, and
 *   PP_ERR_CAPACITY if some rank's 2 E_r + 4 S_r words exceed words_per_rank (its rows would be read from the
 *   next rank's row, or past the buffer); PP_ERR_ARG for an odd words_per_rank, world outside 1..64 or an empty
 *   rank range.  Nothing is written when the call refuses.
 *   cuda_stream != NULL: the kernel is only enqueued on that stream (the caller synchronises with it; the copy-out
 *   of one step's tables then overlaps the upload of the next step's trace -- opposite PCIe directions).  The two
 *   capacity refusals are then not reported, since the call does not wait for the kernel: it writes nothing, and
 *   the caller sizes the tables and words_per_rank from the records. */
typedef struct pp_unpacked_tables {
    int64_t cap_events, cap_segments;
    int64_t *ev_start, *ev_len;
    int64_t *seg_event, *seg_start, *seg_end;
    double *mean, *std, *min, *max;
} pp_unpacked_tables;
int pp_unpack_tables(pp_ctx *ctx, const int64_t *dev_gathered, int world, int64_t words_per_rank,
                     const int64_t *dev_records, const pp_unpacked_tables *out, int out_is_host, void *cuda_stream);
/* The same for the rows of the ranks [rank_lo, rank_hi) only, written from index 0 of the tables (event ids and
 * event starts stay global).  With one process per GPU every rank copies out the rows of its own chunk
 * (rank_lo = rank, rank_hi = rank + 1): the result reaches host memory over all the GPUs' links at once, the way
 * the trace went up. */
int pp_unpack_tables_range(pp_ctx *ctx, const int64_t *dev_gathered, int world, int64_t words_per_rank,
                           const int64_t *dev_records, int rank_lo, int rank_hi, const pp_unpacked_tables *out,
                           int out_is_host, void *cuda_stream);
int pp_pack_tables(pp_ctx *ctx, const int64_t *dev_records, int rank, int64_t sample_offset, int64_t *dev_out,
                   int64_t cap_words);

#ifdef __cplusplus
}
#endif
#endif
