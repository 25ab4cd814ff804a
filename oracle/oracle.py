"""Python face of the CPU oracle (TEST INFRASTRUCTURE, see oracle/__init__.py).

Functions cite the reference lines they restate (paths relative to
/root/reference).  Heavy loops live in ``pypore_oracle.c`` (ctypes); the numpy
calls the reference itself makes (np.mean/np.std/np.min/np.max,
scipy.signal.bessel) are made here the same way.
"""
import ctypes
import importlib.machinery
import importlib.util
import math
import os
import sys
import types

import numpy as np

from . import build_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

_i64p = ctypes.POINTER(ctypes.c_int64)
_i32p = ctypes.POINTER(ctypes.c_int)
_f64p = ctypes.POINTER(ctypes.c_double)


def _p(arr, typ):
    return arr.ctypes.data_as(typ) if arr is not None else None


def lib():
    global _lib
    if _lib is None:
        path = build_oracle.build_port()
        L = ctypes.CDLL(path)
        L.orc_threshold_tics.restype = ctypes.c_int64
        L.orc_threshold_tics.argtypes = [_f64p, ctypes.c_int64, ctypes.c_double, _i64p, ctypes.c_int64]
        L.orc_run_minmax.restype = None
        L.orc_run_minmax.argtypes = [_f64p, _i64p, ctypes.c_int64, _f64p, _f64p]
        L.orc_cumsum.restype = None
        L.orc_cumsum.argtypes = [_f64p, ctypes.c_int64, _f64p, _f64p]
        L.orc_statsplit.restype = ctypes.c_int
        L.orc_statsplit.argtypes = [_f64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_double, _i32p, ctypes.c_int, _i64p, _f64p, _f64p]
        L.orc_window_gains.restype = None
        L.orc_window_gains.argtypes = [_f64p, _f64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _f64p]
        L.orc_statsplit_events.restype = ctypes.c_int
        L.orc_statsplit_events.argtypes = [_f64p, _i64p, _i64p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_double, _i32p, _i64p, _i32p, _i64p,
                                           ctypes.c_int]
        L.orc_filtfilt.restype = ctypes.c_int
        L.orc_filtfilt.argtypes = [_f64p, _f64p, _f64p, ctypes.c_int, _f64p, ctypes.c_int64, _f64p]
        _lib = L
    return _lib


def _f64(x):
    return np.ascontiguousarray(x, dtype=np.float64)


# --------------------------------------------------------------------------
# FastStatSplit.__init__: PyPore/cparsers.pyx:55-101
# --------------------------------------------------------------------------
def min_gain(min_width=100, max_width=1000000, window_width=10000, min_gain_per_sample=None,
             false_positive_rate=None, prior_segments_per_second=None, sampling_freq=1.e5,
             cutoff_freq=None):
    """The gain threshold FastStatSplit derives from its arguments.

    Raises AssertionError on the same conditions (cparsers.pyx:69-76).  The C
    ints of cparsers.pyx:51 truncate like ``int()``.
    """
    mw, MW, W, fs = int(min_width), int(max_width), int(window_width), int(sampling_freq)
    if not false_positive_rate:
        false_positive_rate = sampling_freq
    if not prior_segments_per_second:
        prior_segments_per_second = sampling_freq / 2.
    assert MW >= mw
    assert W >= 2 * mw
    if cutoff_freq:
        assert cutoff_freq <= 0.5 * sampling_freq
    if min_gain_per_sample:
        g = min_gain_per_sample * W
    else:
        k = cutoff_freq / (0.5 * sampling_freq) if cutoff_freq else 1
        sps = prior_segments_per_second
        g = (-math.log(sps / (sampling_freq - sps)) - math.log(false_positive_rate / sampling_freq)) / k
    return g * 2


# --------------------------------------------------------------------------
# lambda_event_parser: PyPore/parsers.py:131-155
# --------------------------------------------------------------------------
def threshold_runs(trace, threshold):
    """Runs on either side of the threshold: (start[int64], length[int64], min, max, below[bool])."""
    x = _f64(trace)
    n = x.shape[0]
    if n == 0:
        z = np.zeros(0, np.int64)
        return z, z.copy(), np.zeros(0), np.zeros(0), np.zeros(0, bool)
    cap = 1024
    while True:
        tics = np.empty(cap, np.int64)
        k = lib().orc_threshold_tics(_p(x, _f64p), n, float(threshold), _p(tics, _i64p), cap)
        if k >= 0:
            break
        cap *= 8
    tics = tics[:k].copy()
    mn = np.empty(k - 1)
    mx = np.empty(k - 1)
    lib().orc_run_minmax(_p(x, _f64p), _p(tics, _i64p), k, _p(mn, _f64p), _p(mx, _f64p))
    start = tics[:-1]
    length = np.diff(tics)
    below = x[start] < threshold
    return start, length, mn, mx, below


class _RunProxy(object):
    """What a rule sees of a piece (SURVEY App. A.1 item 6): duration, start, min, max, n, current."""

    def __init__(self, x, start, n, mn, mx):
        self.start, self.duration, self.n, self.min, self.max = start, n, n, mn, mx
        self._x = x

    @property
    def current(self):
        return self._x[self.start:self.start + self.n]

    @property
    def mean(self):
        return np.mean(self.current)

    @property
    def std(self):
        return np.std(self.current)


def select_runs(trace, runs, rules):
    """_lambda_select (parsers.py:136-140): keep pieces for which ALL rules hold."""
    x = _f64(trace)
    start, length, mn, mx, _ = runs
    keep = []
    for i in range(len(start)):
        ev = _RunProxy(x, int(start[i]), int(length[i]), mn[i], mx[i])
        if np.all([rule(ev) for rule in rules]):
            keep.append(i)
    return np.asarray(keep, dtype=np.int64)


def default_rules(threshold):
    """The default rule list of parsers.py:133-135."""
    return [lambda e: e.duration > 100000, lambda e: e.min > -0.5, lambda e: e.max < threshold]


def events(trace, threshold, rules=None):
    """(start, length) in samples of the events File.parse would create (DataTypes.py:595-600)."""
    runs = threshold_runs(trace, threshold)
    keep = select_runs(trace, runs, rules if rules else default_rules(threshold))
    return runs[0][keep], runs[1][keep]


# --------------------------------------------------------------------------
# FastStatSplit.parse: PyPore/cparsers.pyx:103-203
# --------------------------------------------------------------------------
def cumsum(x):
    x = _f64(x)
    c = np.empty_like(x)
    c2 = np.empty_like(x)
    lib().orc_cumsum(_p(x, _f64p), x.shape[0], _p(c, _f64p), _p(c2, _f64p))
    return c, c2


def statsplit(event, min_width=100, max_width=1000000, window_width=10000, gain=None,
              return_info=False, **gain_kwargs):
    """Breakpoints (event-relative samples, sorted) of FastStatSplit.parse on one event.

    ``gain`` overrides the min_gain derived from ``gain_kwargs``.  Segments are
    the consecutive pairs of [0] + breakpoints + [len] (cparsers.pyx:115-116).
    """
    x = _f64(event)
    if gain is None:
        gain = min_gain(min_width, max_width, window_width, **gain_kwargs)
    n = x.shape[0]
    cap = n // max(int(min_width), 1) + 4
    bp = np.empty(cap, np.int32)
    st = np.zeros(2, np.int64)
    gains = np.empty(cap) if return_info else None
    margins = np.empty(cap) if return_info else None
    k = lib().orc_statsplit(_p(x, _f64p), n, int(min_width), int(max_width), int(window_width),
                            float(gain), _p(bp, _i32p), cap, _p(st, _i64p),
                            _p(gains, _f64p), _p(margins, _f64p))
    if k < 0:
        raise RuntimeError("oracle statsplit overflow")
    if return_info:
        return bp[:k].astype(np.int64), dict(ncand=int(st[0]), nscan=int(st[1]),
                                             gains=gains[:k].copy(), margins=margins[:k].copy())
    return bp[:k].astype(np.int64)


def margin_audit(event, min_width=100, max_width=1000000, window_width=10000, gain=None, **gain_kwargs):
    """Smallest decision margins of FastStatSplit.parse on one event (SURVEY section 4):
    (best - runner-up over the scans that split, min_gain - best over those that did not, number of scans)."""
    x = _f64(event)
    if gain is None:
        gain = min_gain(min_width, max_width, window_width, **gain_kwargs)
    out = np.zeros(3)
    f = lib().orc_statsplit_audit
    f.restype = ctypes.c_int
    f.argtypes = [_f64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, _f64p]
    if f(_p(x, _f64p), x.shape[0], int(min_width), int(max_width), int(window_width), float(gain),
         _p(out, _f64p)) != 0:
        raise RuntimeError("oracle audit overflow")
    return float(out[0]), float(out[1]), int(out[2])


def _window_gains(c, c2, start, end, first, last):
    out = np.empty(max(last - first + 1, 0))
    if out.shape[0]:
        lib().orc_window_gains(_p(c, _f64p), _p(c2, _f64p), int(start), int(end), int(first), int(last),
                               _p(out, _f64p))
    return out


def _sequential_best(gains, min_gain, first):
    """`if gain > min_gain: min_gain = gain; x = i` over the candidates in order (cparsers.pyx:149-151,
    238-240): the first occurrence of the largest gain above the threshold; NaN never wins."""
    best, x = min_gain, -1
    for j, g in enumerate(gains):
        if g > best:
            best, x = g, first + j
    return float(best), x


def best_single_split(event):
    """FastStatSplit.best_single_split (cparsers.pyx:120-155): window [0, len-1), candidates
    2 .. len-4, threshold 0.  Returns (gain, index)."""
    x = _f64(event)
    c, c2 = cumsum(x)
    end = x.shape[0] - 1
    if end - 2 <= 2:
        return 0., -1
    return _sequential_best(_window_gains(c, c2, 0, end, 2, end - 3), 0., 2)


def score_samples(event, no_split=False, min_width=100, max_width=1000000, window_width=10000, gain=None,
                  **gain_kwargs):
    """FastStatSplit.score_samples (cparsers.pyx:205-275): one length-len(event) score array per window
    scan in recursion order, or list(scores of the single scan of [0, len)) with no_split."""
    x = _f64(event)
    if gain is None:
        gain = min_gain(min_width, max_width, window_width, **gain_kwargs)
    mw, MW, W = int(min_width), int(max_width), int(window_width)
    c, c2 = cumsum(x)
    L = x.shape[0]

    def stepwise_score(start, end):           # _best_split_stepwise_score, cparsers.pyx:217-241
        if end - start <= 2 * mw:
            return -1, []
        g = _window_gains(c, c2, start, end, start + mw, end - mw)
        score = np.zeros(L)
        score[start + mw:end + 1 - mw] = g
        return _sequential_best(g, gain, start + mw)[1], score

    def rec(start, end, no_split):            # _recursive_split_scoring, cparsers.pyx:243-275
        scores, split_at = [], -1
        if no_split:
            return list(stepwise_score(start, end)[1])
        for pseudostart in range(start, end - 2 * mw, W // 2):
            if pseudostart > start + MW:
                split_at = min(start + MW, end - mw)
                return scores + rec(split_at, end, 0)
            pseudoend = min(end, pseudostart + W)
            split_at, score = stepwise_score(pseudostart, pseudoend)
            scores.append(score)
            if split_at >= 0:
                break
        if split_at == -1:
            if end - start <= MW:
                return scores
            split_at = min(start + MW, end - mw)
        return scores + rec(start, split_at, 0) + rec(split_at, end, 0)

    return rec(0, L, no_split)


EPS_PER_SAMPLE, EPS_CONST = 3.6e-7, 1e-6   # the device's screening error bound (split.cuh K3_EPS_*), nats


def scan_log(event, min_width=100, max_width=1000000, window_width=10000, gain=None, **gain_kwargs):
    """One record per window scan of FastStatSplit.parse (cparsers.pyx:157-203), in the C oracle's arithmetic.

    Walks the recursion like score_samples (explicit stack: any order gives the same scans).  Each record is a dict:
    ps, pe, x (the split, -1 for none: first occurrence of the largest gain above min_gain, NaN never wins), best /
    best_i (largest non-NaN gain, first occurrence; -inf / -1 if every gain is NaN), second / second_i (largest
    non-NaN gain at another candidate), n_nan, n_posinf, n_near (candidates within 2 eps(n) of best, eps(n) =
    n * EPS_PER_SAMPLE + EPS_CONST) and gains (every candidate ps+mw .. pe-mw).  Also returns the breakpoints,
    sorted, and the work counters (ncand, nscan) of statsplit(return_info=True)."""
    x = _f64(event)
    if gain is None:
        gain = min_gain(min_width, max_width, window_width, **gain_kwargs)
    mw, MW, W = int(min_width), int(max_width), int(window_width)
    c, c2 = cumsum(x)
    log, bps = [], []
    stack = [(0, x.shape[0])]
    while stack:
        start, end = stack.pop()
        split_at, forced_right = -1, False
        for ps in range(start, end - 2 * mw, W // 2):
            if ps > start + MW:
                split_at, forced_right = min(start + MW, end - mw), True
                break
            pe = min(end, ps + W)
            if pe - ps <= 2 * mw:
                continue
            g = _window_gains(c, c2, ps, pe, ps + mw, pe - mw)
            r = dict(ps=ps, pe=pe, x=_sequential_best(g, gain, ps + mw)[1], gains=g)
            ok = ~np.isnan(g)
            r["n_nan"] = int((~ok).sum())
            r["n_posinf"] = int(np.isposinf(g).sum())
            r["best"], r["best_i"], r["second"], r["second_i"], r["n_near"] = -np.inf, -1, -np.inf, -1, 0
            if ok.any():
                j = int(np.argmax(np.where(ok, g, -np.inf)))
                if not ok[j]:
                    j = int(np.flatnonzero(ok)[0])
                r["best"], r["best_i"] = float(g[j]), ps + mw + j
                rest = ok.copy()
                rest[j] = False
                if rest.any():
                    k = int(np.argmax(np.where(rest, g, -np.inf)))
                    if not rest[k]:
                        k = int(np.flatnonzero(rest)[0])
                    r["second"], r["second_i"] = float(g[k]), ps + mw + k
                n = pe - ps
                with np.errstate(invalid="ignore"):
                    r["n_near"] = int((g[ok] >= r["best"] - 2 * (n * EPS_PER_SAMPLE + EPS_CONST)).sum())
            log.append(r)
            split_at = r["x"]
            if split_at >= 0:
                break
        if forced_right:
            bps.append(split_at)
            stack.append((split_at, end))
            continue
        if split_at == -1:
            if end - start <= MW:
                continue
            split_at = min(start + MW, end - mw)
        bps.append(split_at)
        stack.append((split_at, end))
        stack.append((start, split_at))
    ncand = int(sum(len(r["gains"]) for r in log))
    return log, np.sort(np.asarray(bps, np.int64)), dict(ncand=ncand, nscan=len(log))


def statsplit_events(trace, ev_start, ev_len, min_width=100, max_width=1000000, window_width=10000,
                     gain=None, threads=1, **gain_kwargs):
    """FastStatSplit over many events of one float64 trace.

    Returns (seg_event, seg_start, seg_end, ncand): flat segment table with
    event-relative sample indices, ordered by (event, start).
    """
    x = _f64(trace)
    ev_start = np.ascontiguousarray(ev_start, np.int64)
    ev_len = np.ascontiguousarray(ev_len, np.int64)
    if gain is None:
        gain = min_gain(min_width, max_width, window_width, **gain_kwargs)
    E = ev_start.shape[0]
    caps = ev_len // max(int(min_width), 1) + 4
    off = np.zeros(E + 1, np.int64)
    np.cumsum(caps, out=off[1:])
    bp = np.empty(max(int(off[-1]), 1), np.int32)
    nbp = np.zeros(max(E, 1), np.int32)
    ncand = ctypes.c_int64(0)
    r = lib().orc_statsplit_events(_p(x, _f64p), _p(ev_start, _i64p), _p(ev_len, _i64p), E,
                                   int(min_width), int(max_width), int(window_width), float(gain),
                                   _p(bp, _i32p), _p(off, _i64p), _p(nbp, _i32p),
                                   ctypes.byref(ncand), int(threads))
    if r < 0:
        raise RuntimeError("oracle statsplit overflow")
    seg_event, seg_start, seg_end = [], [], []
    for e in range(E):
        b = bp[off[e]:off[e] + nbp[e]].astype(np.int64)
        edges = np.concatenate(([0], b, [ev_len[e]]))
        seg_event.append(np.full(len(edges) - 1, e, np.int64))
        seg_start.append(edges[:-1])
        seg_end.append(edges[1:])
    if E == 0:
        z = np.zeros(0, np.int64)
        return z, z.copy(), z.copy(), 0
    return (np.concatenate(seg_event), np.concatenate(seg_start), np.concatenate(seg_end),
            int(ncand.value))


# --------------------------------------------------------------------------
# Segment.mean/std/min/max: PyPore/core.py:209-223 (numpy over the float64 view)
# --------------------------------------------------------------------------
def segment_stats(x, starts, ends):
    x = _f64(x)
    n = len(starts)
    out = np.empty((4, n))
    for i in range(n):
        v = x[int(starts[i]):int(ends[i])]
        out[0, i] = np.mean(v)
        out[1, i] = np.std(v)
        out[2, i] = np.min(v)
        out[3, i] = np.max(v)
    return out[0], out[1], out[2], out[3]


# --------------------------------------------------------------------------
# Event.filter: PyPore/DataTypes.py:258-274 (scipy.signal.bessel + filtfilt)
# --------------------------------------------------------------------------
def bessel_ba(order, cutoff, second):
    """Coefficients exactly as DataTypes.py:268-270 requests them from scipy."""
    from scipy import signal
    nyquist = second / 2.
    b, a = signal.bessel(order, cutoff / nyquist, btype='low', analog=0, output='ba')
    return _f64(b), _f64(a)


def lfilter_zi(b, a):
    """Steady-state DF2T state for a unit step (scipy.signal.lfilter_zi restated)."""
    b = _f64(b)
    a = _f64(a)
    if a[0] != 1.0:
        b = b / a[0]
        a = a / a[0]
    n = max(len(a), len(b))
    a = np.r_[a, np.zeros(n - len(a))]
    b = np.r_[b, np.zeros(n - len(b))]
    comp = np.zeros((n - 1, n - 1))
    comp[0, :] = -a[1:]
    for i in range(1, n - 1):
        comp[i, i - 1] = 1.0
    IminusA = np.eye(n - 1) - comp.T
    B = b[1:] - a[1:] * b[0]
    return np.linalg.solve(IminusA, B)


def filtfilt(b, a, x):
    """scipy.signal.filtfilt(b, a, x) with default padding, restated in C (SURVEY App. A.5)."""
    b = _f64(b)
    a = _f64(a)
    x = _f64(x)
    nc = max(len(a), len(b))
    padlen = 3 * nc
    if x.shape[0] <= padlen:
        raise ValueError("The length of the input vector x must be greater than padlen, which is %d."
                         % padlen)
    bb = np.r_[b, np.zeros(nc - len(b))] / a[0]
    aa = np.r_[a, np.zeros(nc - len(a))] / a[0]
    zi = _f64(lfilter_zi(bb, aa))
    out = np.empty_like(x)
    r = lib().orc_filtfilt(_p(bb, _f64p), _p(aa, _f64p), _p(zi, _f64p), nc, _p(x, _f64p), x.shape[0],
                           _p(out, _f64p))
    if r != 0:
        raise RuntimeError("oracle filtfilt failed")
    return out


def event_filter(x, second, order=1, cutoff=2000.):
    b, a = bessel_ba(order, cutoff, second)
    return filtfilt(b, a, x)


# --------------------------------------------------------------------------
# The compiled reference (oracle/_ref): the unmodified cparsers.pyx
# --------------------------------------------------------------------------
_ref_mod = None


class _StubSegment(object):
    """Stand-in for PyPore.core.Segment so the compiled reference can build its
    return list on a box without /root/reference.  Holds what
    cparsers.pyx:115-116 passes: current view, start, duration, end."""

    def __init__(self, current, **kwargs):
        self.current = current
        for k, v in kwargs.items():
            setattr(self, k, v)


def ref_available():
    build_oracle.build_ref()
    return os.path.exists(build_oracle.ref_so_path())


def load_ref_cparsers():
    """Import the reference's compiled cparsers module from oracle/_ref (SURVEY App. B)."""
    global _ref_mod
    if _ref_mod is not None:
        return _ref_mod
    so = build_oracle.build_ref()
    if not so or not os.path.exists(so):
        raise RuntimeError("oracle/_ref is not built and /root/reference is absent")
    import itertools
    if not hasattr(itertools, "izip"):
        itertools.izip = zip  # cparsers.pyx:17 is Python-2 source
    saved_core = sys.modules.get("core")
    saved_pkg = sys.modules.get("PyPore")
    core = types.ModuleType("core")
    core.Segment = _StubSegment
    pkg = types.ModuleType("PyPore")
    pkg.__path__ = [os.path.dirname(so)]
    sys.modules["core"] = core
    sys.modules["PyPore"] = pkg
    sys.modules["PyPore.core"] = core
    try:
        loader = importlib.machinery.ExtensionFileLoader("PyPore.cparsers", so)
        spec = importlib.util.spec_from_file_location("PyPore.cparsers", so, loader=loader)
        mod = importlib.util.module_from_spec(spec)
        loader.exec_module(mod)
    finally:
        # do not leave stub modules behind for unrelated imports
        for name, saved in (("core", saved_core), ("PyPore", saved_pkg)):
            if saved is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = saved
        sys.modules.pop("PyPore.core", None)
    _ref_mod = mod
    return mod
