"""Cases for the streamed host pipeline (pp_pipeline_host, pp_pipeline_host_tables, pp_pipeline_host_adc16), shared by
tests/test_gpu_streamed.py (device against the resident run and the oracle) and tests/test_streamed_cases_cpu.py (every
case still reaches what it was built for).

The streamed call copies the trace in chunks of `chunk_samples` rounded up to K1_TILE and, per chunk, runs every stage
over the events completed so far.  A run is complete once the scan has seen the first sample after it, so the run
ending at sample e (exclusive) is finished by the chunk that holds sample e, and the trace's last run only by the final
chunk.  `completions` restates that, so that the CPU test can tell which chunk completes which event."""
import functools
import os

import numpy as np

import oracle
from pypore_b200 import synth
from pypore_b200.adc import AdcTrace

K1_TILE = 4096           # threshold.cuh: chunk sizes are rounded up to a multiple of this
K2_TILE = 2048           # prefix.cuh: tile of the multi-CTA prefix scan of long events
K2F_MAX_LEN = 32768      # prefix.cuh: longest event one warp scans
K3_CAP = 10240           # split.cuh: longer events are walked by k3_spine first
SEL_THREADS = 1024       # threshold.cuh: runs k1_select_events examines per trip
DEFAULT_CHUNK = 16 << 20
PREFIX_AUTO, PREFIX_SEQUENTIAL, PREFIX_PARALLEL = 0, 1, 2

RULES7 = dict(threshold=110.0, rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
SPLITS = {"default": dict(min_width=100, max_width=1000000, window_width=10000),
          "psps10": dict(min_width=100, max_width=1000000, window_width=10000, prior_segments_per_second=10),
          "forced": dict(min_width=50, max_width=2500, window_width=1000),
          "dense": dict(min_width=10, max_width=1000000, window_width=40)}

# event bodies of the long-event trace, in order, separated by open channel; the trace ends inside OPEN_LAST
LONG_LAYOUT = (7000, 10241, 8000, 16384, 32768, 6500, 32769, 24 * 2048, 24 * 2048 + 1, 24 * 2048 - 1, 9000, 7000,
               700000, 8000, 20000, 60 * 2048, 250000, 6000, 7000)
OPEN_LAST = 200003
LONG_CHUNKS = (1, 4095, 4096, 4096 * 37 + 1, 65536, 1 << 20)
TARGET_CHUNKS = (65536, 4096 * 37 + 1)    # the chunkings the long-event targets are asserted for
EDGE_CHUNK = 65536


def rounded(chunk):
    """The chunk size pipeline_host_impl uses for `chunk_samples`."""
    c = chunk if chunk > 0 else DEFAULT_CHUNK
    return -(-c // K1_TILE) * K1_TILE


def streams(n, chunk):
    """True when a trace of n samples is streamed (not run resident) at this chunk size."""
    return rounded(chunk) < n


def chunk_count(n, chunk):
    return -(-n // rounded(chunk))


def completions(n, chunk, start, length):
    """Index of the chunk that completes each run (start, length) of a trace of n samples."""
    end = np.asarray(start, np.int64) + np.asarray(length, np.int64)
    k = chunk_count(n, chunk)
    return np.where(end >= n, k - 1, np.minimum(end // rounded(chunk), k - 1))


def rule_lambdas(rules):
    """The reference's rule list equivalent to a device rule mask (lambda_event_parser: every rule must hold)."""
    m = rules["rule_mask"]
    out = []
    if m & 1:
        out.append(lambda e: e.duration > rules["duration_gt"])
    if m & 8:
        out.append(lambda e: e.duration < rules["duration_lt"])
    if m & 2:
        out.append(lambda e: e.min > rules["min_gt"])
    if m & 4:
        out.append(lambda e: e.max < rules["max_lt"])
    return out or [lambda e: True]


class Case(object):
    """A trace (float32 or AdcTrace), the rules, the split parameters, the chunk sizes it is streamed with and,
    optionally, device options (option id -> value) and a prefix mode."""

    def __init__(self, name, x, rules=RULES7, split="default", chunks=(EDGE_CHUNK,), options=None,
                 prefix_mode=PREFIX_AUTO, oracle_key=None):
        self.name, self.x, self.rules, self.split = name, x, dict(rules), split
        self.chunks, self.options, self.prefix_mode = tuple(chunks), dict(options or {}), prefix_mode
        self.oracle_key = oracle_key or name   # cases on the same current with the same parameters share one oracle

    @property
    def n(self):
        return len(self.x)

    def current(self):
        return self.x.decode() if isinstance(self.x, AdcTrace) else np.asarray(self.x, np.float64)

    def split_params(self):
        kw = dict(SPLITS[self.split])
        mw, MW, W = kw.pop("min_width"), kw.pop("max_width"), kw.pop("window_width")
        return mw, MW, W, oracle.min_gain(mw, MW, W, **kw)

    def pipeline_kw(self):
        mw, MW, W, gain = self.split_params()
        return dict(self.rules, min_width=mw, max_width=MW, window_width=W, min_gain=gain,
                    prefix_mode=self.prefix_mode)


def oracle_runs(case):
    """(runs, indices of the runs the rules select) of the oracle on the case's current."""
    x = case.current()
    runs = oracle.threshold_runs(x, case.rules["threshold"])
    return runs, oracle.select_runs(x, runs, rule_lambdas(case.rules))


def oracle_tables(case):
    """What the pipeline must give: event (start, length), segment (event, start, end) and segment statistics."""
    x = case.current()
    runs, keep = oracle_runs(case)
    ws, wl = runs[0][keep], runs[1][keep]
    mw, MW, W, gain = case.split_params()
    se, ss, sn, _ = oracle.statsplit_events(x, ws, wl, mw, MW, W, gain=gain, threads=os.cpu_count() or 1)
    base = ws[se] if len(se) else np.zeros(0, np.int64)
    m, sd, mn, mx = oracle.segment_stats(x, base + ss, base + sn)
    return dict(ev_start=ws, ev_len=wl, event=se, start=ss, end=sn, mean=m, std=sd, min=mn, max=mx)


# ---------------------------------------------------------------------------------------------------------------
# traces
# ---------------------------------------------------------------------------------------------------------------
def _gap(rng, n, tier="A"):
    g = rng.normal(synth.OPEN_MEAN, synth.OPEN_STD, n).astype(np.float32)
    return synth.quantise(g) if tier == "A" else g


@functools.lru_cache(maxsize=None)
def long_trace(tier):
    """Short tier-A/B events mixed with every length class of the split stages (LONG_LAYOUT), open channel between
    them; the trace ends inside a long event (the open last run).  About 1.7 M samples."""
    rng = np.random.RandomState(71 if tier == "A" else 72)
    parts = []
    for i, L in enumerate(LONG_LAYOUT + (OPEN_LAST,)):
        parts.append(_gap(rng, int(rng.randint(3000, 5000)), tier))
        parts.append(synth.make_long_event(L, seed=500 + i, tier=tier))
    x = np.concatenate(parts)
    x.setflags(write=False)
    return x


def _paint(x, a, b, seed):
    x[a:b] = synth.make_long_event(b - a, seed=seed, tier="A")


@functools.lru_cache(maxsize=None)
def edge_trace():
    """Open channel with events and non-finite samples placed on the boundaries b = k * EDGE_CHUNK, and one sample
    in the last chunk (n = 12 * EDGE_CHUNK + 1)."""
    C = EDGE_CHUNK
    n = 12 * C + 1
    x = _gap(np.random.RandomState(81), n)
    _paint(x, C, C + 8000, 1)                   # a crossing exactly at b
    _paint(x, 2 * C + 1, 2 * C + 7000, 2)       # ... at b + 1
    _paint(x, 3 * C - 1, 3 * C + 6000, 3)       # ... at b - 1
    _paint(x, 4 * C - 9000, 4 * C, 4)           # an event whose last sample is b - 1
    _paint(x, 5 * C - 5000, 5 * C + 5000, 5)    # NaN / +inf at the last / first sample of a chunk inside an event
    x[5 * C - 1], x[5 * C] = np.nan, np.inf
    _paint(x, 6 * C - 5000, 6 * C + 5000, 6)    # -inf at both (below the threshold: the event goes on)
    x[6 * C - 1], x[6 * C] = -np.inf, -np.inf
    x[7 * C - 1], x[7 * C] = np.nan, -np.inf    # the same inside the open channel
    x[8 * C - 1], x[8 * C] = np.inf, np.nan
    _paint(x, 9 * C - 4000, 9 * C + 4000, 9)    # a run whose minimum is the first sample of a chunk
    x[9 * C] = 5.0
    x[10 * C] = 200.0                           # ... an open-channel run whose maximum is
    _paint(x, 11 * C - 4000, 11 * C + 4000, 11)  # ... an event whose maximum is
    x[11 * C] = 105.0
    _paint(x, 12 * C - 3000, n, 12)             # the last event is open and completed by a 1-sample chunk
    x.setflags(write=False)
    return x


@functools.lru_cache(maxsize=None)
def dense_trace():
    """~50-sample events from sample 30001 on for 140,000 samples: a 65,536-sample chunk completes more than 1,024
    runs, starting at a run index that is not a multiple of 1,024, while the whole trace stays within the run table
    the streamed call reserves (n / 256 + 4096 runs)."""
    rng = np.random.RandomState(91)
    n = 400000
    x = _gap(rng, n)
    i = np.arange(140000)
    below = (i // 50) % 2 == 0
    seg = np.where(below, 50.0 + (i % 7) * 0.125, 120.0 + (i % 5) * 0.25).astype(np.float32)
    x[30001:30001 + 140000] = seg
    x.setflags(write=False)
    return x


def overflow_trace():
    """A crossing every 50 samples: 24,000 runs, more than the n / 256 + 4096 the streamed call reserves, so
    pp_pipeline_host redoes the whole trace resident (test_host_tables_too_small_fall_back_to_downloads's shape)."""
    n = 1200000
    x = np.where((np.arange(n) // 50) % 2 == 0, 50.0, 120.0).astype(np.float32)
    x += (np.arange(n) % 7).astype(np.float32) * 0.125
    return x


DENSE_RULES = dict(threshold=110.0, rule_mask=5, duration_gt=20, duration_lt=0, min_gt=0.0, max_lt=110.0)


@functools.lru_cache(maxsize=None)
def rule_trace():
    """Open channel first (the run at sample 0 is above the threshold), tier-A events of 3,000..12,000 samples, one
    open-channel gap holding a NaN, and the trace ends in the open channel (the open last run is above)."""
    rng = np.random.RandomState(61)
    parts = [_gap(rng, 5000)]
    for i in range(40):
        parts.append(synth.make_long_event(int(rng.randint(3000, 12000)), seed=700 + i))
        g = _gap(rng, int(rng.randint(2000, 6000)))
        if i == 17:
            g[len(g) // 2] = np.nan
        parts.append(g)
    x = np.concatenate(parts)
    x.setflags(write=False)
    return x


def rule_sets():
    """name -> rules: every mask shape, durations at an actual event length and +-1, min_gt at an actual minimum."""
    runs = oracle.threshold_runs(rule_trace().astype(np.float64), 110.0)
    start, length, mn, mx, below = runs
    ev = np.flatnonzero(below)
    L = int(length[ev[7]])
    m = float(mn[ev[11]])
    base = dict(threshold=110.0, duration_gt=0, duration_lt=0, min_gt=0.0, max_lt=0.0)
    out = {"mask0": dict(base, rule_mask=0),
           "mask1_1000": dict(base, rule_mask=1, duration_gt=1000),
           "mask2_all": dict(base, rule_mask=2, min_gt=-0.5),
           "mask2_at_min": dict(base, rule_mask=2, min_gt=m),
           "mask4": dict(base, rule_mask=4, max_lt=110.0),
           "mask7": dict(RULES7),
           "mask15": dict(base, rule_mask=15, duration_gt=1000, duration_lt=L + 1, min_gt=-0.5, max_lt=110.0)}
    for d in (-1, 0, 1):
        out["mask1_at_len%+d" % d] = dict(base, rule_mask=1, duration_gt=L + d)
        out["mask9_at_len%+d" % d] = dict(base, rule_mask=9, duration_gt=1000, duration_lt=L + d)
    return out


def adc_of(x32, scale, offset=0.0, extremes=()):
    """The counts whose decoding is closest to x32; `extremes` = sample indices that get -32768, 32767 in turn."""
    c = np.round((np.asarray(x32, np.float64) - offset) / scale)
    c = np.clip(c, -32768, 32767).astype(np.int16)
    for j, i in enumerate(extremes):
        c[i] = -32768 if j % 2 == 0 else 32767
    return AdcTrace(c, scale, offset)


ADC_SOURCES = {"adc_1_32": (1.0 / 32, 0.0), "adc_real": (0.0305, 0.0123), "adc_negative": (-1.0 / 32, 0.0)}
OPTIONS = {"screen_off": {0: 0}, "flow": {3: 1}, "ctas1": {2: 1}, "ctas3": {2: 3}, "spine_off": {1: 0}}


def long_chunks(n):
    """Every chunking of the long-event traces: the fixed sizes, the largest multiple of K1_TILE below n (a short
    last chunk) and n itself (the resident fallback)."""
    return LONG_CHUNKS + ((n - 1) // K1_TILE * K1_TILE, n)


@functools.lru_cache(maxsize=None)
def cases():
    """name -> Case (built lazily: traces are made on first use)."""
    out = {}
    for tier in ("A", "B"):
        x = long_trace(tier)
        out["long_" + tier] = Case("long_" + tier, x, chunks=long_chunks(len(x)))
    xa = long_trace("A")
    for split in ("psps10", "forced"):
        out["long_A_" + split] = Case("long_A_" + split, xa, split=split, chunks=TARGET_CHUNKS)
    for name, opts in OPTIONS.items():
        out["option_" + name] = Case("option_" + name, xa, chunks=TARGET_CHUNKS, options=opts, oracle_key="long_A")
    for tier in ("A", "B"):
        for mode, mname in ((PREFIX_SEQUENTIAL, "sequential"), (PREFIX_PARALLEL, "parallel")):
            out["prefix_%s_%s" % (mname, tier)] = Case("prefix_%s_%s" % (mname, tier), long_trace(tier),
                                                       chunks=TARGET_CHUNKS, prefix_mode=mode,
                                                       oracle_key="long_" + tier)
    for name, (scale, offset) in ADC_SOURCES.items():
        ext = [k * EDGE_CHUNK + d for k in (3, 7, 11, 19) for d in (-1, 0)]
        out[name] = Case(name, adc_of(xa, scale, offset, ext), chunks=TARGET_CHUNKS)
    xe = edge_trace()
    for rname, rules in (("mask7", RULES7), ("mask0", dict(RULES7, rule_mask=0))):
        out["edges_" + rname] = Case("edges_" + rname, xe, rules=rules, chunks=(EDGE_CHUNK, 4096, 32768))
    out["dense"] = Case("dense", dense_trace(), rules=DENSE_RULES, split="dense", chunks=(EDGE_CHUNK, 4096 * 13 + 1))
    for rname, rules in rule_sets().items():
        out["rules_" + rname] = Case("rules_" + rname, rule_trace(), rules=rules, chunks=(EDGE_CHUNK, 4096 * 37 + 1))
    return out


# ---------------------------------------------------------------------------------------------------------------
# the public path: one trace longer than the default chunk
# ---------------------------------------------------------------------------------------------------------------
BIG_LONG = 1200000        # the event across sample DEFAULT_CHUNK
BIG_OPEN = 1000000        # the open last event


@functools.lru_cache(maxsize=None)
def big_trace():
    """~18.4 M samples of open channel with 60 short tier-A events in the first 15 M, a 1.2 M-sample event across
    sample 16 * 2**20 and a 1 M-sample event the trace ends in (streamed by File.parse in two default chunks)."""
    rng = np.random.RandomState(101)
    a = DEFAULT_CHUNK - BIG_LONG // 2
    n = a + BIG_LONG + 4000 + BIG_OPEN
    x = _gap(rng, n)
    for i, s in enumerate(np.linspace(5000, 15000000, 60).astype(np.int64)):
        _paint(x, int(s), int(s) + int(rng.randint(3000, 12000)), 900 + i)
    _paint(x, a, a + BIG_LONG, 990)
    _paint(x, n - BIG_OPEN, n, 991)
    x.setflags(write=False)
    return x


def hmm_model(S=6, seed=2):
    """S states over the levels of the synthetic events, sticky transitions, some forbidden ones."""
    from pypore_b200.hmm import HMM
    rng = np.random.default_rng(seed)
    mean = np.sort(rng.uniform(0.0, 110.0, S))
    std = rng.uniform(1.0, 6.0, S)
    trans = rng.uniform(0.0, 1.0, (S, S))
    trans[rng.uniform(size=(S, S)) < 0.2] = 0.0
    np.fill_diagonal(trans, 4.0)
    return HMM(mean, std, trans, starts=rng.uniform(0.1, 1.0, S))
