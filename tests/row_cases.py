"""Cases for the row locality of K3c + K4 (compaction and segment statistics), shared by tests/test_gpu_rows.py (device
against itself, the exact references and the oracle) and tests/test_row_cases_cpu.py (every case reaches what it was
built for).

The contract: a row's statistics depend only on its own samples and on where they sit in the trace or the flat event
space -- not on the other rows, on the row range of the launch or on the length of the table.  K4 sums a row in G
strided lanes and G sets the order of the fp64 sums, so G must follow from the row alone.  The cases put rows into
tables whose mean row length (`total / rows`, the quantity a per-launch width would follow) lies on the other side of
K4_WIDE = 512 than in another run over the same rows: a streamed export's early or inner chunks, a subset of the
events, the table after an HMM merge.  Their samples are order-sensitive (fp64 sums of non-dyadic values), so that
another width would show in the last bits.

Every segment is a clean level step: levels far apart against the noise, so that the split search puts every
breakpoint where it was placed.  A segment whose draw the oracle splits otherwise is drawn again (`designed_event`)."""
import functools

import numpy as np

import oracle
from pypore_b200.adc import AdcTrace

K4_WIDE = 512             # stats.cuh: rows of at least this many samples are summed by 32 lanes, shorter ones by 8
K4_ONE_PASS = 65536       # stats.cuh: longer rows take two passes
CP_BLOCK_SAMPLES = 32768  # split.cuh: one k3c compaction block (1024 bitmap words)
CP_SCAN_BLOCKS = 1024     # split.cuh: k3c_scan covers this many blocks per trip
K1_TILE = 4096

ADC_SCALE, ADC_OFFSET = 0.0305, 0.0123
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
GAIN = oracle.min_gain(prior_segments_per_second=10, **SPLIT)
# duration and max rules only: float32 levels sit near 0
RULES = dict(threshold=110.0, rule_mask=5, duration_gt=100, duration_lt=0, min_gt=0.0, max_lt=110.0)
OPEN_MEAN, OPEN_STD = 120.0, 1.5


def width(total, rows):
    """The group width a launch over `rows` rows of `total` samples picked from their mean length (the rule the row
    contract replaces)."""
    return 8 if total // rows < K4_WIDE else 32


def rounded(chunk):
    return -(-chunk // K1_TILE) * K1_TILE


# ---------------------------------------------------------------------------------------------------------------
# events of designed level steps
# ---------------------------------------------------------------------------------------------------------------
def _levels(rng, k, kind):
    """k levels, neighbours at least 20 apart.  float32 data alternate between levels near 0 (where float32 samples
    have fine last bits, so that the fp64 sums of their squares round) and levels of 30..60."""
    if kind == "float32":
        return [rng.uniform(-1.0, 1.0) if i % 2 == 0 else rng.uniform(30.0, 60.0) for i in range(k)]
    out = [rng.uniform(10.0, 90.0)]
    while len(out) < k:
        v = rng.uniform(10.0, 90.0)
        if abs(v - out[-1]) >= 20.0:
            out.append(v)
    return out


def _body(rng, seglens, kind, levels=None, noise=1.0):
    lv = levels if levels is not None else _levels(rng, len(seglens), kind)
    x = np.concatenate([v + rng.normal(0.0, noise, L) for v, L in zip(lv, seglens)])
    if kind == "float32":
        return x.astype(np.float32).astype(np.float64)
    if kind == "adc":
        return np.round((x - ADC_OFFSET) / ADC_SCALE) * ADC_SCALE + ADC_OFFSET
    return x


def designed_event(seed, seglens, kind, levels=None, noise=1.0, split=SPLIT, gain=GAIN):
    """(samples as float64, breakpoints) of one event of level steps that the oracle splits exactly at the steps."""
    want = np.cumsum(seglens)[:-1]
    for attempt in range(50):
        rng = np.random.RandomState(seed * 100 + attempt)
        x = _body(rng, seglens, kind, levels, noise)
        bp = oracle.statsplit(x, split["min_width"], split["max_width"], split["window_width"], gain=gain)
        if np.array_equal(bp, want):
            return x, want
    raise AssertionError("no draw of event %d splits at its steps" % seed)


def _seglens(rng, k, lo, hi):
    return [int(v) for v in rng.randint(lo, hi + 1, k)]


# ---------------------------------------------------------------------------------------------------------------
# traces for the threshold pipeline (resident and streamed)
# ---------------------------------------------------------------------------------------------------------------
class Trace(object):
    """A float64 current with designed events: `x` (float32 current or AdcTrace, what the pipeline reads), `x64`
    (the decoded current), event (start, length) and per event the designed breakpoints."""

    def __init__(self, x, x64, ev_start, ev_len, bps):
        self.x, self.x64 = x, x64
        self.ev_start, self.ev_len = np.asarray(ev_start, np.int64), np.asarray(ev_len, np.int64)
        self.bps = bps

    @property
    def n(self):
        return len(self.x64)

    def table(self):
        """The designed segment table: event, start, end (event-relative)."""
        e, s, t = [], [], []
        for i, (L, b) in enumerate(zip(self.ev_len, self.bps)):
            edges = np.r_[0, b, L]
            e.append(np.full(len(edges) - 1, i, np.int64))
            s.append(edges[:-1])
            t.append(edges[1:])
        return np.concatenate(e), np.concatenate(s), np.concatenate(t)


def _stream_trace(blocks, kind, seed):
    """blocks = [(n_events, segments per event, segment length lo, hi, gap lo, hi)]: open channel, then the events of
    every block in turn, each followed by open channel."""
    rng = np.random.RandomState(seed)
    parts = [rng.normal(OPEN_MEAN, OPEN_STD, 1500)]
    pos = 1500
    starts, lens, bps = [], [], []
    ev = 0
    for n_ev, k, lo, hi, glo, ghi in blocks:
        for _ in range(n_ev):
            x, b = designed_event(seed * 1000 + ev, _seglens(rng, k, lo, hi), kind)
            ev += 1
            starts.append(pos)
            lens.append(len(x))
            bps.append(b)
            parts.append(x)
            g = int(rng.randint(glo, ghi + 1))
            parts.append(rng.normal(OPEN_MEAN, OPEN_STD, g))
            pos += len(x) + g
    x64 = np.concatenate(parts)
    if kind == "float32":
        x32 = x64.astype(np.float32)
        return Trace(x32, x32.astype(np.float64), starts, lens, bps)
    c = np.clip(np.round((x64 - ADC_OFFSET) / ADC_SCALE), -32768, 32767).astype(np.int16)
    a = AdcTrace(c, ADC_SCALE, ADC_OFFSET)
    return Trace(a, a.decode(), starts, lens, bps)


LONG_BLOCK = (3, 5, 2000, 3000, 9000, 10000)     # ~12,500-sample events, segments averaging 2,500, apart
SHORT_BLOCK = (50, 12, 130, 170, 1000, 1500)     # ~1,800-sample events, segments averaging 150


@functools.lru_cache(maxsize=None)
def long_then_short(kind):
    """First chunk of 65,536 samples: only events of segments >= 2,000 samples; then many events stepping every
    ~150 samples, so that the whole table averages < 256 samples per row."""
    return _stream_trace([LONG_BLOCK, SHORT_BLOCK], kind, 11 if kind == "float32" else 12)


@functools.lru_cache(maxsize=None)
def short_long_short(kind):
    """Short rows, a block of long ones that lifts the running mean past 512 at an inner chunk, short rows again."""
    return _stream_trace([(10, 10, 130, 170, 800, 1200), (5, 5, 2000, 3000, 1500, 2500), (45, 10, 130, 170, 800, 1200)],
                         kind, 13 if kind == "float32" else 14)


STREAM_CASES = {"long_then_short": (long_then_short, (65536, 4096 * 7, 4096 * 20 + 1)),
                "short_long_short": (short_long_short, (32768, 4096 * 5 + 1))}
STREAM_KINDS = ("float32", "adc")


def completed_by(trace, chunk):
    """Per chunk of the streamed call: the events that end before the chunk's last sample (completed by then
    whatever the chunk-edge rules finalise)."""
    C = rounded(chunk)
    k = -(-trace.n // C)
    end = trace.ev_start + trace.ev_len
    return [np.flatnonzero(end < (c + 1) * C) for c in range(k)]


def chunk_widths(trace, chunk):
    """The width a per-launch rule picks in each chunk's launch (running totals), and for the resident launch."""
    seg_per_ev = np.array([len(b) + 1 for b in trace.bps], np.int64)
    out = []
    for done in completed_by(trace, chunk):
        if len(done):
            out.append(width(int(trace.ev_len[done].sum()), int(seg_per_ev[done].sum())))
        else:
            out.append(None)
    return out, width(int(trace.ev_len.sum()), int(seg_per_ev.sum()))


# ---------------------------------------------------------------------------------------------------------------
# placed events (set_events) and their subsets
# ---------------------------------------------------------------------------------------------------------------
class Placed(object):
    """Events placed on a float64 or int16 trace, NaN (ADC: the int16 extremes) between them.  `rows` = the events'
    float64 samples, `bps` their designed breakpoints, `start` their trace positions."""

    def __init__(self, kind, rows, bps, seed):
        rng = np.random.RandomState(seed)
        self.kind, self.rows, self.bps = kind, rows, bps
        pos, starts = 0, []
        for r in rows:
            pos += int(rng.randint(1, 10))
            starts.append(pos)
            pos += len(r)
        self.start = np.array(starts, np.int64)
        self.length = np.array([len(r) for r in rows], np.int64)
        self.n = pos + 9
        if kind == "adc":
            c = np.full(self.n, 32767, np.int16)
            c[::2] = -32768
            for s, r in zip(starts, rows):
                c[s:s + len(r)] = np.round((r - ADC_OFFSET) / ADC_SCALE).astype(np.int16)
            self.trace = AdcTrace(c, ADC_SCALE, ADC_OFFSET)
            self.x64 = self.trace.decode()
        else:
            self.trace = np.full(self.n, np.nan)
            for s, r in zip(starts, rows):
                self.trace[s:s + len(r)] = r
            self.x64 = self.trace

    def upload(self, ctx, which):
        if self.kind == "adc":
            ctx.upload_trace_adc16(self.trace)
        else:
            ctx.upload_trace_f64(self.trace)
        ctx.set_events(self.start[which], self.length[which])

    def table(self, which):
        """Designed segment table of the events `which`: event (index into `which`), start, end."""
        e, s, t = [], [], []
        for i, j in enumerate(which):
            edges = np.r_[0, self.bps[j], self.length[j]]
            e.append(np.full(len(edges) - 1, i, np.int64))
            s.append(edges[:-1])
            t.append(edges[1:])
        return np.concatenate(e), np.concatenate(s), np.concatenate(t)


N_LONG_EVENTS, N_SHORT_EVENTS = 6, 400


@functools.lru_cache(maxsize=None)
def subset_events(kind):
    """6 events of five ~2,500-sample segments, then 400 events of 300 samples in two segments: all events average
    < 512 samples per segment and per event, the long ones alone far more."""
    rows, bps = [], []
    for i in range(N_LONG_EVENTS):
        x, b = designed_event(3000 + i, [2500 + 37 * i, 2300, 2700 - 11 * i, 2450, 2600], kind)
        rows.append(x)
        bps.append(b)
    for i in range(N_SHORT_EVENTS):
        x, b = designed_event(4000 + i, [150 + i % 7, 150 - i % 5], kind)
        rows.append(x)
        bps.append(b)
    return Placed(kind, rows, bps, 21 if kind == "float64" else 22)


def subsets():
    """name -> indices of the events uploaded (always in trace order)."""
    n = N_LONG_EVENTS + N_SHORT_EVENTS
    return {"all": np.arange(n), "long": np.arange(N_LONG_EVENTS),
            "long_plus_one_short": np.r_[np.arange(N_LONG_EVENTS), N_LONG_EVENTS + 123]}


SUBSET_KINDS = ("float64", "adc")


# ---------------------------------------------------------------------------------------------------------------
# HMM merge: pairs of near levels that one state covers
# ---------------------------------------------------------------------------------------------------------------
MERGE_STATES = (20.0, 45.0, 70.0, 95.0)
MERGE_PATTERN = ((0, 2), (1, 2), (2, 1), (3, 2), (0, 2))   # (state, segments) per run of one state
N_MERGE_EVENTS = 40


def merge_model():
    from pypore_b200.hmm import HMM
    S = len(MERGE_STATES)
    trans = np.full((S, S), 1.0)
    np.fill_diagonal(trans, 3.0)
    return HMM(list(MERGE_STATES), [4.0] * S, trans)


@functools.lru_cache(maxsize=None)
def merge_events(kind):
    """Events of ~320-sample segments in runs of one state: pairs at the state's mean -+ 1.5 (split apart: the step is
    10 noise deviations) and singles.  Before the merge rows average < 512 samples; after it, > 512."""
    rows, bps = [], []
    for i in range(N_MERGE_EVENTS):
        rng = np.random.RandomState(5000 + i)
        levels, lens = [], []
        for j, (s, k) in enumerate(MERGE_PATTERN):
            off = (-1.5, 1.5) if (i + j) % 2 == 0 else (1.5, -1.5)
            levels += [MERGE_STATES[s] + off[q] for q in range(k)] if k == 2 else [MERGE_STATES[s]]
            lens += _seglens(rng, k, 290, 350)
        x, b = designed_event(6000 + i, lens, kind, levels=levels, noise=0.15)
        rows.append(x)
        bps.append(b)
    return Placed(kind, rows, bps, 31 if kind == "float64" else 32)


def merged_table(p):
    """The designed table after the merge: runs of one state become one segment."""
    e, s, t = [], [], []
    for i, (L, b) in enumerate(zip(p.length, p.bps)):
        edges = np.r_[0, b, L]
        k = 0
        for _, n in MERGE_PATTERN:
            e.append(i)
            s.append(edges[k])
            t.append(edges[k + n])
            k += n
    return np.array(e, np.int64), np.array(s, np.int64), np.array(t, np.int64)


# ---------------------------------------------------------------------------------------------------------------
# compaction edges on packed float64 events (upload_events_f64: flat offsets are the running lengths)
# ---------------------------------------------------------------------------------------------------------------
EDGE_SPLIT = dict(min_width=10, max_width=1000000, window_width=1000)
EDGE_GAIN = oracle.min_gain(prior_segments_per_second=1e-4, **EDGE_SPLIT)
BIG_SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
BIG_GAIN = oracle.min_gain(prior_segments_per_second=1e-4, **BIG_SPLIT)
ALT_SPLIT = dict(min_width=1, max_width=1000000, window_width=8)
ALT_GAIN = oracle.min_gain(**ALT_SPLIT)


def _flat_events(marks, n, seed, tiny=(), noise=1e-3):
    """Events covering flat [0, n): `marks` = flat positions where an event starts ("e") or a breakpoint sits ("b");
    `tiny` = (flat start, length) of events too short to split.  Piecewise-constant levels 20 apart with small noise.
    Returns (events as float64 arrays, designed flat breakpoints = every event start and breakpoint)."""
    rng = np.random.RandomState(seed)
    cuts = sorted(set([0] + [f for f, _ in marks] + [f for f, _ in tiny] + [f + L for f, L in tiny]))
    kinds = dict(marks)
    kinds.update({f: "e" for f, _ in tiny})
    for f, L in tiny:
        kinds.setdefault(f + L, "e")
    kinds[0] = "e"
    cuts = [c for c in cuts if c < n]
    events, cur, lv = [], [], 50.0
    for a, b in zip(cuts, cuts[1:] + [n]):
        if kinds.get(a, "b") == "e" and cur:
            events.append(np.concatenate(cur))
            cur = []
        lv = 30.0 if lv > 40.0 else 70.0
        cur.append(lv + rng.normal(0.0, noise, b - a))
    events.append(np.concatenate(cur))
    return events, np.array(cuts, np.int64)


@functools.lru_cache(maxsize=None)
def compaction_edges():
    """Flat event space of 3.5 blocks: event starts and breakpoints on bit 0 and bit 31 of bitmap words, on both sides
    of block edges (a 1-sample event holds the last sample of block 2), events of 1, 2 and 3 samples."""
    B = CP_BLOCK_SAMPLES
    marks = [(4096 + 31, "e"), (4096 + 64, "b"), (8192 + 32 * 5 + 31, "b"), (8192 + 32 * 9, "e"),
             (B - 1, "b"), (B + 40, "e"), (2 * B, "b"), (2 * B + 63, "b"), (2 * B + 5000, "e"),
             (3 * B + 500, "b"), (3 * B + 1000 + 31, "e")]
    tiny = [(12000, 1), (12001, 2), (12003, 3), (20000, 3), (3 * B - 1, 1), (3 * B, 2)]
    return _flat_events(marks, 3 * B + B // 2, 41, tiny)


@functools.lru_cache(maxsize=None)
def alternating_events():
    """min_width = 1 over samples alternating between two exact levels: every sample of a word is a breakpoint."""
    x = np.where(np.arange(1000) % 2 == 0, 10.0, 20.0)
    y = np.where(np.arange(777) % 2 == 0, -5.0, 5.0)
    return [x, np.full(33, 7.0), y]


BIG_BLOCKS = CP_SCAN_BLOCKS + 13


@functools.lru_cache(maxsize=None)
def big_flat_events():
    """More than 1,024 compaction blocks (> 33,554,432 flat samples): k3c_scan carries its running offset across
    trips.  Events of ~1 M samples with a step every ~4,000 samples, marks on both sides of the 1,024-block edge."""
    B = CP_BLOCK_SAMPLES
    n = BIG_BLOCKS * B + 777
    rng = np.random.RandomState(43)
    marks = []
    f = 0
    while f < n - 8000:
        f += int(rng.randint(3000, 5000))
        marks.append((f, "e" if rng.uniform() < 0.01 else "b"))
    E = CP_SCAN_BLOCKS * B
    marks = [m for m in marks if abs(m[0] - E) > 200]
    marks += [(E - 1, "b"), (E + 100, "e"), (E + 287, "b")]    # bits 31 | 4, 31 of the words there
    marks = sorted(m for m in marks if m[0] < n - 100)
    return _flat_events(marks, n, 44, noise=1e-2)


def flat_offsets(events):
    return np.r_[0, np.cumsum([len(e) for e in events])].astype(np.int64)


def oracle_flat(events, split, gain):
    """The oracle's segment table of packed events: event, start, end, and the flat starts."""
    off = flat_offsets(events)
    x = np.concatenate(events)
    e, s, t, _ = oracle.statsplit_events(x, off[:-1], np.diff(off), split["min_width"], split["max_width"],
                                         split["window_width"], gain=gain, threads=8)
    return e, s, t, off[e] + s


# ---------------------------------------------------------------------------------------------------------------
# order sensitivity: a model of the orders G lanes sum in
#
# This approximates K4's order: it puts element j in lane j % G and adds plain products.  K4 gives each lane whole
# 16-byte vectors (element j in lane (j / N) % G, shifted by the row's 16-byte phase) and accumulates d*d with fma.
# The model only answers whether a row's sums depend on their order at all, which is what the cases need; that the
# device's sums actually change with the width is shown on the GPU (tests/test_gpu_rows.py fails under a per-launch
# width on these cases).
# ---------------------------------------------------------------------------------------------------------------
def lane_sums(d, G):
    """sum(d) and sum(d*d) with element j in lane j % G, each lane in order, then the xor butterfly of K4."""
    m = -(-len(d) // G) * G
    a = np.zeros(m)
    a[:len(d)] = d
    a = a.reshape(-1, G)
    s1, s2 = np.zeros(G), np.zeros(G)
    for r in a:
        s1 = s1 + r
        s2 = s2 + r * r
    idx = np.arange(G)
    step = G // 2
    while step:
        s1 = s1 + s1[idx ^ step]
        s2 = s2 + s2[idx ^ step]
        step //= 2
    return s1[0], s2[0]


def order_sensitive(row):
    """True when sequential, 8-lane and 32-lane sums of d = x - x[0] and d*d do not all agree bit for bit (in the
    model above)."""
    d = np.asarray(row, np.float64) - float(row[0])
    s1, s2 = 0.0, 0.0
    for v in d:
        s1 += v
        s2 += v * v
    got = {(s1, s2), lane_sums(d, 8), lane_sums(d, 32)}
    return len(got) > 1
