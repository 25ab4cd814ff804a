"""Cases for the sharded step on one GPU, shared by tests/test_gpu_shard_tables.py (several contexts play the ranks)
and tests/test_shard_cases_cpu.py (every case still reaches the plan shape it was built for).

A case is one float32 global trace cut into contiguous chunks, one per rank, at positions read off the oracle's run
table of that trace, plus the rules and the speculative halo: how many samples of its right neighbour's chunk each
rank finds behind its own before anything is known about the runs (pypore_b200.dist.ShardedPipeline's load())."""
import functools

import numpy as np

import oracle
from pypore_b200 import dist as ppdist
from pypore_b200 import synth

THRESHOLD = 110.0
RULES7 = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
RULES5 = dict(rule_mask=5, duration_gt=1000, duration_lt=0, min_gt=0.0, max_lt=110.0)   # no MIN_GT
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
HALO_SPECULATIVE = 1 << 16
EXTRA_CAPACITY = 1 << 17     # room behind every chunk for the halo, speculative or received


class Case(object):
    """`cuts`: world + 1 sample offsets; `halo`: speculative halo per boundary (capped at the neighbour's chunk);
    `targets`: what the case is built to reach (checked by both test modules):
        joined      boundaries b (between rank b and b + 1) where the two runs join
        covered     boundaries whose straddling event the speculative halo covers (device plan keeps it)
        rejected    boundaries whose joined run the rules reject
        span3       owner rank of an event over three or more chunks
        empty       ranks with no events
        redo        the flags (16, 1) the device-planned step raises
        overflow    ranks whose chunk has more runs than the run table starts with"""

    def __init__(self, name, x, cuts, rules=RULES7, halo=HALO_SPECULATIVE, host_halo=False, **targets):
        self.name, self.x, self.cuts, self.rules = name, x, [int(c) for c in cuts], dict(rules)
        self.halo, self.host_halo = halo, host_halo
        self.targets = dict(joined=(), covered=(), rejected=(), span3=(), empty=(), redo=0, overflow=())
        self.targets.update(targets)

    @property
    def world(self):
        return len(self.cuts) - 1

    @property
    def n(self):
        return len(self.x)

    def chunk(self, r):
        return self.x[self.cuts[r]:self.cuts[r + 1]]

    def lens(self):
        return [self.cuts[r + 1] - self.cuts[r] for r in range(self.world)]

    def halos(self, halo=None):
        """Speculative halo of every rank (0 for the last one)."""
        h = self.halo if halo is None else halo
        lens = self.lens()
        hs = h if isinstance(h, (list, tuple)) else [h] * self.world
        return [int(min(hs[r], lens[r + 1])) if r < self.world - 1 else 0 for r in range(self.world)]


def rule_lambdas(rules):
    """The reference's rule list equivalent to a device rule mask."""
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


def runs(x):
    return oracle.threshold_runs(np.asarray(x, np.float64), THRESHOLD)


def events_of(x, rules=RULES7):
    """(start, length) of the events the oracle selects in x."""
    r = runs(x)
    keep = oracle.select_runs(np.asarray(x, np.float64), r, rule_lambdas(rules))
    return r[0][keep], r[1][keep]


def infos(case):
    """Every rank's boundary record, built from the oracle's runs of its chunk."""
    out = []
    for r in range(case.world):
        c = case.chunk(r)
        s, l, mn, mx, below = runs(c)
        first = (s[0], l[0], mn[0], mx[0], below[0])
        last = (s[-1], l[-1], mn[-1], mx[-1], below[-1])
        out.append(ppdist.boundary_info(len(c), len(s), first, last))
    return np.stack(out)


def plans(case):
    return ppdist.plan_boundaries(infos(case), case.rules)


def need(plan):
    return sum(cnt for _, cnt in plan["recv"])


def _open(n, seed):
    g = np.random.RandomState(seed).normal(synth.OPEN_MEAN, synth.OPEN_STD, n)
    return synth.quantise(g)


# ------------------------------------------------------------------------------------------------------------------
def _one_rank():
    x = synth.make_trace(6, seed=60)
    return Case("w1_whole", x, [0, len(x)])


def _straddle(name, halo_from_need, host_halo=False):
    """Two ranks, the cut 2500 samples inside the fourth event; the halo is 2^16, exactly what the owner needs, or one
    sample short of it (the device plan then asks for the redo)."""
    x = synth.make_trace(8, seed=61)
    ws, wl = events_of(x)
    cut = int(ws[3]) + 2500
    need = int(ws[3] + wl[3]) - cut
    halo = {None: HALO_SPECULATIVE, 0: need, -1: need - 1}[halo_from_need]
    covered = (0,) if halo >= need else ()
    return Case(name, x, [0, cut, len(x)], halo=halo, host_halo=host_halo, joined=(0,), covered=covered,
                redo=0 if covered else 16)


def _event_edges():
    """Three ranks: one cut exactly at an event's first sample, one a sample past another event's last sample."""
    x = synth.make_trace(9, seed=62)
    ws, wl = events_of(x)
    return Case("w3_event_edges", x, [0, int(ws[3]), int(ws[6] + wl[6]), len(x)])


def _open_chunk():
    """Three ranks; rank 1's chunk lies in the open channel between two events, one run above the threshold.  That
    run joins the runs on both sides into one open-channel run over three chunks, which MAX_LT rejects."""
    x = synth.make_trace(6, seed=75)
    ws, wl = events_of(x)
    return Case("w3_open_chunk", x, [0, int(ws[2] + wl[2]) + 500, int(ws[3]) - 500, len(x)], joined=(0, 1),
                rejected=(0,), empty=(1,))


def _span3():
    """Five ranks; rank 2's chunk lies inside one 60,000-sample event that starts in rank 1's chunk and ends in rank
    3's, so rank 1 receives pieces from two ranks.  The other two boundaries cut events the halo covers."""
    a = synth.make_trace(4, seed=63)
    b = synth.make_trace(4, seed=65)
    x = np.concatenate([a, synth.make_long_event(60000, seed=64), b])
    ws, wl = events_of(x)
    L = len(a)
    assert ws[4] == L and wl[4] >= 60000
    cuts = [0, int(ws[2]) + 2000, L + 5000, L + 35000, int(ws[6]) + 3000, len(x)]
    return Case("w5_span3", x, cuts, joined=(0, 1, 2, 3), covered=(0, 3), span3=(1,), empty=(2,), redo=16)


def _rejected():
    """Three ranks, two straddling runs the rules reject: an 800-sample event (too short even joined) across the first
    cut, and an event whose right-hand part holds a sub-zero spike (MIN_GT) across the second.  The middle rank's only
    events are those two, so it has none."""
    x = synth.make_trace(6, seed=66)
    ws, wl = events_of(x)
    g = int(ws[2] + wl[2]) + 1500                        # inside the open channel after the third event
    x[g:g + 800] = synth.make_long_event(800, seed=67)
    cut1 = g + 300
    cut2 = int(ws[3]) + 2000
    x, hit = synth.add_subzero_spikes(x, [cut2], [int(ws[3] + wl[3]) - cut2], frac=1.0, seed=68)
    assert list(hit) == [0]
    return Case("w3_rejected", x, [0, cut1, cut2, len(x)], joined=(0, 1), rejected=(0, 1), empty=(1,))


def _nan_edge():
    """Two ranks; the first sample of rank 1 is a NaN inside an event: NaN counts as above, so the runs do not join
    and the event is two events."""
    x = synth.make_trace(6, seed=69)
    ws, _ = events_of(x)
    cut = int(ws[2]) + 3000
    x[cut] = np.nan
    return Case("w2_nan_edge", x, [0, cut, len(x)])


def _non_finite():
    """Three ranks under a rule mask without MIN_GT: an event with a -inf sample in the halo part of the straddling
    event at the first cut (min = mean = -inf, std = NaN), and -0.0 samples in an event of rank 2 whose other samples
    are all positive (min = -0.0)."""
    x = synth.make_trace(7, seed=70)
    ws, wl = events_of(x, RULES5)
    cut1 = int(ws[2]) + 2500
    x[cut1 + 1000] = -np.inf
    x[int(ws[5]) + 3000] = -0.0
    x[int(ws[5]) + 3001] = -0.0
    cut2 = int(ws[4])
    return Case("w3_non_finite", x, [0, cut1, cut2, len(x)], rules=RULES5, joined=(0,), covered=(0,))


def overflow_block(n=20000, seed=71):
    """Crossings at every sample: n runs of one sample each."""
    hi = _open(n, seed)
    lo = synth.quantise(np.full(n, 100.0))
    return np.where(np.arange(n) % 2 == 0, lo, hi).astype(np.float32)


def _overflow():
    """Two ranks; rank 1's chunk has ~20,000 one-sample runs, more than the n / 256 + 4096 its run table starts with."""
    a = synth.make_trace(3, seed=72)
    b = synth.make_trace(2, seed=73)
    x = np.concatenate([a, overflow_block(), b])
    ws, wl = events_of(x)
    cut = int(ws[1]) + 2500
    return Case("w2_overflow", x, [0, cut, len(x)], joined=(0,), covered=(0,), overflow=(1,), redo=1)


@functools.lru_cache(maxsize=None)
def cases():
    out = [_one_rank(), _straddle("w2_straddle", None), _straddle("w2_halo_at_need", 0),
           _straddle("w2_halo_short", -1, host_halo=True), _event_edges(), _open_chunk(), _span3(), _rejected(),
           _nan_edge(),
           _non_finite(), _overflow()]
    return {c.name: c for c in out}


def f64_trace(seed=74, n_events=8):
    """A float64 trace float32 cannot hold: ADC counts scaled by 0.0305 and offset by 0.0123, and a cut in the open
    channel between two events (no halo needed)."""
    counts = np.round(synth.make_trace(n_events, seed=seed).astype(np.float64) * 32)
    x = counts * 0.0305 + 0.0123
    ws, wl = events_of(x)
    cut = int(ws[3] + wl[3]) + 1000
    return x, [0, cut, len(x)]
