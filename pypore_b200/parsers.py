"""GPU-backed parsers behind the reference's plug-in protocol.

Mirror of PyPore/parsers.py for the hot path: same class names, constructor
arguments, attributes (so ``to_dict``/``to_json``/``from_json`` round-trip,
parsers.py:42-55,97-107) and the duck-typed ``parse(current) -> [Segment]``
contract (parsers.py:57-59).  The arithmetic runs in libpypore_b200.so.
"""
import json
import math

import numpy as np

from . import _lib
from .adc import AdcTrace
from .core import Segment


class parser(object):
    """Base parser protocol (parsers.py:34-107, GUI hooks omitted)."""

    def __init__(self):
        pass

    def __repr__(self):
        return self.to_json()

    def to_dict(self):
        # the reference drops Qt widgets and lambdas by their repr (parsers.py:42-49); a RuleSet is this
        # repository's stand-in for the rule lambdas and is dropped the same way
        d = {key: val for key, val in self.__dict__.items() if key != 'param_dict' and not key.startswith('_')
             if type(val) in (int, float) or (('Qt' not in repr(val)) and 'lambda' not in repr(val)
                                              and not isinstance(val, RuleSet) and not callable(val))}
        d['name'] = self.__class__.__name__
        return d

    def to_json(self, filename=False):
        d = {k: v for k, v in self.to_dict().items() if not callable(v) and not isinstance(v, RuleSet)}
        _json = json.dumps(d, indent=4, separators=(',', ' : '))
        if filename:
            with open(filename, 'w') as out:
                out.write(_json)
        return _json

    def parse(self, current):
        """Default: the whole current as one segment (parsers.py:57-59)."""
        return [Segment(current=current, start=0, duration=current.shape[0] / 100000)]

    @classmethod
    def from_json(cls, _json):
        if _json.endswith(".json"):
            with open(_json, 'r') as infile:
                _json = ''.join(line for line in infile)
        d = json.loads(_json)
        name = d['name']
        del d['name']
        import pypore_b200.parsers as mod
        return getattr(mod, name)(**d)


class MemoryParse(object):
    """Rebuild segments from stored split points (parsers.py:110-122)."""

    def __init__(self, starts, ends):
        self.starts = starts
        self.ends = ends

    def parse(self, current):
        return [Segment(current=np.array(current[int(s):int(e)], copy=True), start=s, duration=(e - s))
                for s, e in zip(self.starts, self.ends)]


# --------------------------------------------------------------------------
# Rules
# --------------------------------------------------------------------------
class RuleSet(list):
    """A list of rule callables that ALSO says what they are, so that
    ``lambda_event_parser`` can evaluate them on the device instead of calling
    Python per run.  Iterating it yields ordinary ``rule(event) -> bool``
    callables, so it is a valid ``rules=`` argument for the reference too."""

    def __init__(self, duration_gt=None, duration_lt=None, min_gt=None, max_lt=None):
        rules = []
        self.mask = 0
        self.duration_gt = self.duration_lt = 0
        self.min_gt = self.max_lt = 0.0
        if duration_gt is not None:
            self.mask |= _lib.RULE_DURATION_GT
            self.duration_gt = duration_gt
            rules.append(lambda event, v=duration_gt: event.duration > v)
        if duration_lt is not None:
            self.mask |= _lib.RULE_DURATION_LT
            self.duration_lt = duration_lt
            rules.append(lambda event, v=duration_lt: event.duration < v)
        if min_gt is not None:
            self.mask |= _lib.RULE_MIN_GT
            self.min_gt = min_gt
            rules.append(lambda event, v=min_gt: event.min > v)
        if max_lt is not None:
            self.mask |= _lib.RULE_MAX_LT
            self.max_lt = max_lt
            rules.append(lambda event, v=max_lt: event.max < v)
        list.__init__(self, rules)

    def device_args(self):
        """Arguments for pp_select_events.  ``duration > v`` on integer sample counts
        equals ``duration > floor(v)``; ``duration < v`` equals ``duration < ceil(v)``."""
        def whole(v, rounding):
            # +-inf (and anything beyond int64) clamps to the int64 limits: the comparison's outcome is the same
            v = float(v)
            if v != v:
                raise ValueError("a duration rule cannot be NaN")
            return int(rounding(max(min(v, 9.2e18), -9.2e18)))
        return dict(rule_mask=self.mask,
                    duration_gt=whole(self.duration_gt, math.floor), duration_lt=whole(self.duration_lt, math.ceil),
                    min_gt=float(self.min_gt), max_lt=float(self.max_lt))


class _RunProxy(object):
    """What a rule sees of one piece (SURVEY App. A.1 item 6): ``duration``, ``start``,
    ``min``, ``max``, ``n`` from the device run table; ``current``/``mean``/``std`` lazily (``current`` of an
    AdcTrace: the decoded slice)."""

    def __init__(self, host_current, start, n, mn, mx):
        self.start, self.duration, self.n, self.min, self.max = start, n, n, mn, mx
        self._host = host_current
        self.copy = True  # the stray attribute of parsers.py:152

    @property
    def current(self):
        return self._host[self.start:self.start + self.n]

    @property
    def mean(self):
        return Segment(self.current).mean

    @property
    def std(self):
        return Segment(self.current).std


class lambda_event_parser(parser):
    """Threshold event detector (parsers.py:124-155).

    Events are maximal runs of samples strictly below ``threshold`` (compared in
    float64) that satisfy every rule.  ``rules`` may be any list of callables on
    an event-like object (evaluated on the host against the device run table) or
    a ``RuleSet`` (evaluated on the device).  ``rules=None`` gives the reference
    defaults: duration > 100000 samples, min > -0.5, max < threshold.
    """

    def __init__(self, threshold=90, rules=None):
        self.threshold = threshold
        self._builtin_rules = [lambda event: event.duration > 100000,
                               lambda event: event.min > -0.5,
                               lambda event: event.max < self.threshold]
        self.rules = rules or self._builtin_rules

    def _device_rules(self):
        """The rules as a device-evaluable RuleSet, or None (arbitrary callables: evaluated on the host).  The
        reference's defaults qualify only while ``rules`` still IS the list built in __init__ -- assigning
        ``parser.rules = [...]`` afterwards, which the reference supports, takes effect like any other list."""
        rules = self.rules
        if rules is self.__dict__.get("_builtin_rules"):
            return RuleSet(duration_gt=100000, min_gt=-0.5, max_lt=self.threshold)
        return rules if isinstance(rules, RuleSet) else None

    def _lambda_select(self, events):
        return [event for event in events if np.all([rule(event) for rule in self.rules])]

    # -- device-side helpers shared with File.parse ---------------------------
    def _detect(self, ctx, host_current):
        """Threshold scan + selection on a resident trace.  Returns (start, length,
        min, max) arrays of the selected events (samples)."""
        n_runs = ctx.threshold_scan(self.threshold)
        rs = self._device_rules()
        if rs is not None:
            ne, _ = ctx.select_events(**rs.device_args())
            start, length = ctx.events(ne)
            r_start, r_len, r_min, r_max, _ = ctx.runs(n_runs)
            idx = np.searchsorted(r_start, start)
            return start, length, r_min[idx], r_max[idx]
        r_start, r_len, r_min, r_max, _ = ctx.runs(n_runs)
        keep = [i for i in range(n_runs)
                if np.all([rule(_RunProxy(host_current, int(r_start[i]), int(r_len[i]), r_min[i], r_max[i]))
                           for rule in self.rules])]
        keep = np.asarray(keep, dtype=np.int64)
        ctx.set_events(r_start[keep], r_len[keep])
        return r_start[keep], r_len[keep], r_min[keep], r_max[keep]

    def parse(self, current):
        """One Segment per surviving run: ``current`` (a copy; decoded float64 for an AdcTrace), ``start``
        (np.int64 sample index) and ``duration`` (samples) -- no ``end``, like the reference."""
        host = current if isinstance(current, AdcTrace) else np.asarray(current)
        if host.shape[0] == 0:
            return []
        ctx = _lib.default_context()
        _upload_trace(ctx, host)
        start, length, mn, mx = self._detect(ctx, host)
        out = []
        for s, n in zip(start, length):
            seg = Segment(current=np.array(host[int(s):int(s) + int(n)]), copy=True, start=s, duration=int(n))
            out.append(seg)
        return out


def _device_trace(x):
    """The array handed to the device for a trace given as `x`: float32 input as it is; float64 input as
    float32 when that loses nothing (half the bytes, identical results: double(x32) == x), as float64
    otherwise -- the reference's own loader yields int16 counts times a float64 scale (read_abf.py:208-210),
    which in general is not float32-representable; integer input is exact in float64."""
    x = np.asarray(x)
    if x.dtype == np.float32:
        return np.ascontiguousarray(x)
    if x.dtype.kind in "iub":
        x = x.astype(np.float64)
    if x.dtype != np.float64:
        raise TypeError("trace must be float32, float64 or an integer type, got %s" % x.dtype)
    x32 = x.astype(np.float32)
    if np.array_equal(x32.astype(np.float64), x, equal_nan=True):
        return x32
    return np.ascontiguousarray(x)


def _upload_trace(ctx, x):
    """`x` (any accepted dtype, or an AdcTrace) resident on `ctx`; returns what went up."""
    if isinstance(x, AdcTrace):
        ctx.upload_trace_adc16(x)
        return x
    dev = _device_trace(x)
    if dev.dtype == np.float32:
        ctx.upload_trace(dev)
    else:
        ctx.upload_trace_f64(dev)
    return dev


def _run_pipeline(ctx, x, threshold, **kw):
    """pp_pipeline for a host trace of any accepted dtype: float32 traces and AdcTraces stream through the chunked
    host call, float64 ones are uploaded whole (8 B per sample) and run resident."""
    if isinstance(x, AdcTrace):
        return ctx.pipeline(threshold, host_trace=x, **kw)
    dev = _device_trace(x)
    if dev.dtype == np.float32:
        return ctx.pipeline(threshold, host_trace=dev, **kw)
    ctx.upload_trace_f64(dev)
    return ctx.pipeline(threshold, **kw)


# --------------------------------------------------------------------------
# Segmenter
# --------------------------------------------------------------------------
def statsplit_min_gain(min_width=100, max_width=1000000, window_width=10000, min_gain_per_sample=None,
                       false_positive_rate=None, prior_segments_per_second=None, sampling_freq=1.e5,
                       cutoff_freq=None):
    """FastStatSplit.__init__ (cparsers.pyx:55-101): validation and the gain threshold.

    Returns (min_width, max_width, window_width, min_gain) with the C-int
    truncation of cparsers.pyx:51.
    """
    mw, MW, W = int(min_width), int(max_width), int(window_width)
    fs = int(sampling_freq)  # stored as a C int; the gain formula uses the Python value
    del fs
    if not false_positive_rate:
        false_positive_rate = sampling_freq
    if not prior_segments_per_second:
        prior_segments_per_second = sampling_freq / 2.
    assert MW >= mw, "Maximum width must be greater than minimum width."
    assert W >= 2 * mw, "Window width must be greater than twice the minimum width."
    if cutoff_freq:
        assert cutoff_freq <= 0.5 * sampling_freq, \
            "Cutoff freq must be less than half the sampling frequency."
    if min_gain_per_sample:
        gain = min_gain_per_sample * W
    else:
        k = cutoff_freq / (0.5 * sampling_freq) if cutoff_freq else 1
        sps = prior_segments_per_second
        gain = (-math.log(sps / (sampling_freq - sps)) - math.log(false_positive_rate / sampling_freq)) / k
    return mw, MW, W, gain * 2


def _first_best(gains, min_gain, first_index):
    """The sequential `if gain > best: best = gain; x = i` loop of the reference over an array of
    gains: (best gain, index of its FIRST occurrence), or (min_gain, -1).  NaN never wins."""
    ok = gains > min_gain
    if not ok.any():
        return min_gain, -1
    best = gains[ok].max()
    return float(best), int(first_index + np.flatnonzero(gains == best)[0])


class SpeedyStatSplit(parser):
    """Recursive maximum-likelihood changepoint segmenter (parsers.py:505-528,
    cparsers.pyx:45-203) on the GPU."""

    def __init__(self, min_width=100, max_width=1000000, window_width=10000,
                 min_gain_per_sample=None, false_positive_rate=None,
                 prior_segments_per_second=None, sampling_freq=1.e5, cutoff_freq=None):
        self.min_width = min_width
        self.max_width = max_width
        self.min_gain_per_sample = min_gain_per_sample
        self.window_width = window_width
        self.prior_segments_per_second = prior_segments_per_second
        self.false_positive_rate = false_positive_rate
        self.sampling_freq = sampling_freq
        self.cutoff_freq = cutoff_freq

    def _params(self):
        mw, MW, W, gain = statsplit_min_gain(
            self.min_width, self.max_width, self.window_width, self.min_gain_per_sample,
            self.false_positive_rate, self.prior_segments_per_second, self.sampling_freq, self.cutoff_freq)
        if W // 2 == 0:
            raise ValueError("range() arg 3 must not be zero")  # what the reference's xrange raises
        return mw, MW, W, gain

    @property
    def min_gain(self):
        return self._params()[3]

    def parse(self, current):
        """Segments of one event: ``current`` views, ``start``/``end``/``duration`` in
        samples (cparsers.pyx:115-116), statistics precomputed on the device."""
        return self.parse_many([current])[0]

    @staticmethod
    def _as_event(current):
        cur = np.asarray(current)
        if cur.dtype != np.float64:
            # the reference assigns np.cumsum(current) to a double[:] memoryview (cparsers.pyx:53,110)
            raise ValueError("Buffer dtype mismatch, expected 'double' but got '%s'" %
                             {np.dtype(np.float32): 'float'}.get(cur.dtype, str(cur.dtype)))
        return np.ascontiguousarray(cur)

    def best_single_split(self, current):
        """(gain, index) of the single best split of `current` (parsers.py:530-534 -> cparsers.pyx:120-155):
        window [0, len-1), candidates 2 .. len-4, threshold 0, lowest index on ties; (0.0, -1) if no
        candidate has a positive gain.  Exact reference arithmetic for every candidate on the device."""
        # the reference builds a FastStatSplit first -- WITHOUT cutoff_freq (parsers.py:531-533): same assertions
        statsplit_min_gain(self.min_width, self.max_width, self.window_width, self.min_gain_per_sample,
                           self.false_positive_rate, self.prior_segments_per_second, self.sampling_freq)
        cur = self._as_event(current)
        end = cur.shape[0] - 1
        if end - 4 < 1:  # xrange(2, end-2) is empty
            return 0., -1
        ctx = _lib.default_context()
        ctx.upload_events_f64([cur])
        ctx.prefix()
        gains = ctx.window_gains(0, [0], [end], 2)[0][:end - 4]   # candidates 2 .. end-3
        return _first_best(gains, 0., 2)

    def score_samples(self, current, no_split=False):
        """One length-len(current) score array per window scan, in the reference's recursion order
        (cparsers.pyx:205-275 score_samples / _recursive_split_scoring); no_split=True: the scores of the
        single scan of [0, len) as a plain list.  Exact reference arithmetic on the device, one batched
        call per recursion depth; the recursion itself is replayed on the host."""
        mw, MW, W, min_gain = self._params()
        cur = self._as_event(current)
        L = cur.shape[0]
        ctx = _lib.default_context()
        known = {}
        if L > 0:
            ctx.upload_events_f64([cur])
            ctx.prefix()

        def scan(ps, pe, missing):
            """(split, score array) of window [ps, pe) -- _best_split_stepwise_score -- or None if not computed yet."""
            if pe - ps <= 2 * mw:
                return -1, []
            if (ps, pe) not in known:
                missing.add((ps, pe))
                return None
            return known[(ps, pe)]

        def walk(start, end, missing):
            """_recursive_split_scoring (cparsers.pyx:246-275); returns None while windows are missing."""
            scores, split_at = [], -1
            for pstart in range(start, end - 2 * mw, W // 2):
                if pstart > start + MW:
                    split_at = min(start + MW, end - mw)
                    rest = walk(split_at, end, missing)
                    return None if rest is None else scores + rest
                r = scan(pstart, min(end, pstart + W), missing)
                if r is None:
                    return None
                split_at, score = r
                scores.append(score)
                if split_at >= 0:
                    break
            if split_at == -1:
                if end - start <= MW:
                    return scores
                split_at = min(start + MW, end - mw)
            left, right = walk(start, split_at, missing), walk(split_at, end, missing)
            return None if left is None or right is None else scores + left + right

        def compute(windows):
            windows = sorted(windows)
            gains = ctx.window_gains(0, [w[0] for w in windows], [w[1] for w in windows], mw)
            for (ps, pe), g in zip(windows, gains):
                score = np.zeros(L)
                score[ps + mw:ps + mw + g.shape[0]] = g
                known[(ps, pe)] = (_first_best(g, min_gain, ps + mw)[1], score)

        if no_split:
            missing = set()
            r = scan(0, L, missing)
            if r is None:
                compute(missing)
                r = known[(0, L)]
            return list(r[1])
        while True:
            missing = set()
            out = walk(0, L, missing)
            if out is not None:
                return out
            compute(missing)

    def parse_many(self, currents):
        """Segment many events in one device pass (list of float64 arrays)."""
        mw, MW, W, gain = self._params()
        arrays = []
        for cur in currents:
            cur = np.asarray(cur)
            if cur.dtype != np.float64:
                # FastStatSplit.parse assigns the cumsum to a double[:] memoryview
                raise ValueError("Buffer dtype mismatch, expected 'double' but got '%s'" %
                                 {np.dtype(np.float32): 'float'}.get(cur.dtype, str(cur.dtype)))
            arrays.append(np.ascontiguousarray(cur))
        out = [None] * len(arrays)
        live = [i for i, a in enumerate(arrays) if a.shape[0] > 0]
        for i, a in enumerate(arrays):
            if a.shape[0] == 0:
                out[i] = [Segment(current=a[0:0], start=0, duration=0, end=0)]
        if not live:
            return out
        ctx = _lib.default_context()
        ctx.upload_events_f64([arrays[i] for i in live])
        n_seg = ctx.statsplit(mw, MW, W, gain)
        ctx.segment_stats()
        tab = ctx.segments(n_seg)
        bounds = np.searchsorted(tab["event"], np.arange(len(live) + 1))
        for j, i in enumerate(live):
            a = arrays[i]
            segs = []
            for k in range(bounds[j], bounds[j + 1]):
                s, e = int(tab["start"][k]), int(tab["end"][k])
                seg = Segment(current=a[s:e], start=s, duration=(e - s), end=e)
                seg._set_stats(tab["mean"][k], tab["std"][k], tab["min"][k], tab["max"][k])
                segs.append(seg)
            out[i] = segs
        return out


class FilterDerivativeSegmenter(parser):
    """Filter-derivative segmenter (PyPore/parsers.py:609-656): zero-phase order-1 Bessel low-pass, absolute
    first difference, blocks where it exceeds ``low_threshold``, split points from those blocks.

    Same constructor, attributes and results as the reference, its quirks included: a block is kept when the
    *position* of its largest derivative (``np.argmax``) exceeds ``high_threshold`` (parsers.py:645), and a
    Segment is built for every second pair of split points only (parsers.py:655-656).  The filtfilt -- the
    O(n) arithmetic of the method -- runs on the device through the K5 scan (pp_filter_events, the kernel behind
    Event.filter); the thresholding of the derivative is the reference's own NumPy statements."""

    def __init__(self, low_threshold=1, high_threshold=2, cutoff_freq=1000., sampling_freq=1.e5):
        self.low_threshold = low_threshold
        self.high_threshold = high_threshold
        self.cutoff_freq = cutoff_freq
        self.sampling_freq = sampling_freq

    def parse(self, current):
        from .DataTypes import bessel_coefficients
        x = np.ascontiguousarray(np.array(current), np.float64)
        ctx = _lib.default_context()
        ctx.upload_events_f64([x])
        ctx.filter_events(*bessel_coefficients(1, self.cutoff_freq, self.sampling_freq))   # scipy raises for len <= padlen
        filtered_current = ctx.event_samples(x.shape[0])

        deriv = np.abs(np.diff(filtered_current))
        blocks = np.where(deriv > self.low_threshold, 1, 0)
        block_edges = np.abs(np.diff(blocks))
        tics = np.where(block_edges == 1)[0] + 1

        split_points = [0]
        for start, end in zip(tics[:-1:2], tics[1::2]):
            segment = deriv[start:end]
            if np.argmax(segment) > self.high_threshold:
                split_points = np.concatenate((split_points, [start, end]))
        tics = [int(t) for t in np.concatenate((split_points, [current.shape[0]]))]
        return [Segment(current=current[tics[i]:tics[i + 1]], start=tics[i]) for i in range(0, len(tics) - 1, 2)]
