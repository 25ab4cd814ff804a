"""What a context holds after each call: every download, and every call that reads the prefix sums, answers PP_OK
while its table describes the current events and PP_ERR_STATE once an earlier stage was redone or never ran.  Also
which calls each kind of resident trace (float32, float64, int16 ADC counts) is accepted by."""
import ctypes

import numpy as np
import pytest

from pypore_b200 import _lib, synth
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import bessel_coefficients
from pypore_b200.parsers import statsplit_min_gain

pytestmark = pytest.mark.gpu

OK, ARG, STATE = _lib.PP_OK, _lib.PP_ERR_ARG, _lib.PP_ERR_STATE
RULES = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
FILTER = bessel_coefficients(1, 2000., 1e5)
KINDS = ("float32", "float64", "adc16")


def trace():
    return synth.make_trace(3, seed=31, tier="A")


def put(c, kind, x32):
    if kind == "float32":
        c.upload_trace(x32)
    elif kind == "float64":
        c.upload_trace_f64(x32.astype(np.float64))
    else:
        c.upload_trace_adc16(AdcTrace(np.round(x32.astype(np.float64) * 32).astype(np.int16), 1.0 / 32))


def split(c):
    return c.statsplit(*statsplit_min_gain(**SPLIT))


def codes(c, n):
    """Return code of every download and of the two calls that read the prefix sums; `n` bounds every table and
    every table's total of samples."""
    L, h = c._L, c._h
    f64 = [np.empty(n) for _ in range(5)]
    redone = np.empty(n, np.uint8)
    ps, pe = np.zeros(1, np.int32), np.full(1, 2, np.int32)
    ptr = lambda a: _lib._ptr(a, _lib._f64p)   # noqa: E731
    return dict(
        runs=L.pp_runs_download(h, n, None, None, None, None, None),
        runs_range=L.pp_runs_download_range(h, 0, 0, None, None, None, None, None),
        events=L.pp_events_download(h, n, None, None),
        event_samples=L.pp_event_samples_download(h, n, ptr(f64[0])),
        event_stats=L.pp_event_stats_download(h, n, None, None, None, None),
        segments=L.pp_segments_download(h, n, None, None, None, None, None, None, None),
        segment_stats=L.pp_segments_download(h, n, None, None, None, ptr(f64[1]), None, None, None),
        prefix=L.pp_debug_prefix(h, n, ptr(f64[2]), ptr(f64[3]), _lib._ptr(redone, _lib._u8p)),
        window_gains=L.pp_window_gains(h, 0, 1, _lib._ptr(ps, _lib._i32p), _lib._ptr(pe, _lib._i32p), 1,
                                       ptr(f64[4]), 1),
    )


def expect(runs=False, events=False, samples=False, prefix=False, segments=False, stats=False):
    s = lambda valid: OK if valid else STATE   # noqa: E731
    return dict(runs=s(runs), runs_range=s(runs), events=s(events), event_samples=s(samples),
                event_stats=s(events), segments=s(segments), segment_stats=s(stats), prefix=s(prefix),
                window_gains=s(prefix))


@pytest.mark.parametrize("filtered", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_trace_state_walk(kind, filtered):
    x = trace()
    n = 2 * x.shape[0] + 16    # the appended event overlaps selected ones: more event samples than the trace has
    c = _lib.Context(0)
    try:
        assert codes(c, n) == expect()
        put(c, kind, x)
        assert codes(c, n) == expect()
        assert c.threshold_scan(110.0) > 0
        assert codes(c, n) == expect(runs=True)
        ne, _ = c.select_events(**RULES)
        assert ne > 0
        assert codes(c, n) == expect(runs=True, events=True)
        if filtered:
            c.filter_events(*FILTER)
            assert codes(c, n) == expect(runs=True, events=True, samples=True)
        assert split(c) > 0
        assert codes(c, n) == expect(runs=True, events=True, samples=filtered, prefix=True, segments=True)
        c.segment_stats()
        done = expect(runs=True, events=True, samples=filtered, prefix=True, segments=True, stats=True)
        assert codes(c, n) == done
        if not filtered:
            # a new event: the prefix sums and the segment table no longer describe the event table
            c.append_event(0, 3000)
            assert codes(c, n) == expect(runs=True, events=True)
            split(c)
            assert codes(c, n) == expect(runs=True, events=True, prefix=True, segments=True)
        # a new trace: nothing derived from the old one is left
        put(c, kind, x)
        assert codes(c, n) == expect()
    finally:
        c.close()


def test_uploaded_events_state_walk():
    rng = np.random.RandomState(5)
    arrays = [np.r_[rng.normal(60, 2, 3000), rng.normal(30, 2, 2000)], rng.normal(45, 2, 800),
              np.repeat(rng.uniform(20, 90, 8), 500) + rng.normal(0, 1, 4000)]
    n = sum(len(a) for a in arrays) + 16
    c = _lib.Context(0)
    try:
        c.upload_events_f64(arrays)
        assert codes(c, n) == expect(events=True, samples=True)
        c.filter_events(*FILTER)
        assert codes(c, n) == expect(events=True, samples=True)
        assert split(c) > 0
        assert codes(c, n) == expect(events=True, samples=True, prefix=True, segments=True)
        c.segment_stats()
        assert codes(c, n) == expect(events=True, samples=True, prefix=True, segments=True, stats=True)
        # filtering again changes the events' samples: prefix sums and segments are gone
        c.filter_events(*FILTER)
        assert codes(c, n) == expect(events=True, samples=True)
        split(c)
        assert codes(c, n) == expect(events=True, samples=True, prefix=True, segments=True)
        put(c, "float32", trace())
        assert codes(c, n) == expect()
    finally:
        c.close()


def test_trace_kind_guards():
    """append / extend and the device pointer are for float32 traces only; prefetch, adopt and the sharded calls
    refuse only an ADC trace."""
    x = trace()
    x16 = np.full(16, 120.0, np.float32)
    zeros = np.zeros(8, np.int64)
    c = _lib.Context(0)
    L, h = c._L, c._h
    try:
        assert L.pp_trace_device_ptr(h) is None          # no trace yet
        assert L.pp_trace_append(h, x16.ctypes.data, 0, 0) == STATE
        assert L.pp_trace_extend(h, 0) == STATE
        p, _ = c._params(110.0, **SPLIT, min_gain=0.0, **RULES)
        pf, keep = c._params(110.0, **SPLIT, min_gain=0.0, filter_ba=FILTER, **RULES)   # keep: pf's coefficients
        want = lambda accepted: OK if accepted else STATE   # noqa: E731
        for kind in KINDS:
            f32, not_adc = kind == "float32", kind != "adc16"
            put(c, kind, x)
            c.threshold_scan(110.0)                       # sizes the event buffers used as device scratch below
            ev_start, ev_len = ctypes.c_void_p(c.table_ptr(7)), ctypes.c_void_p(c.table_ptr(8))
            assert (L.pp_trace_device_ptr(h) is not None) == f32, kind
            assert L.pp_trace_append(h, x16.ctypes.data, 0, 0) == want(f32), kind
            assert L.pp_trace_extend(h, 0) == want(f32), kind
            # past the trace check these two refuse the filter (PP_ERR_ARG) before they launch anything
            assert L.pp_shard_finish(h, ctypes.byref(pf), 0, 0, 0, 0, 0, ev_len) == (ARG if not_adc else STATE)
            assert L.pp_shard_finish_planned(h, ctypes.byref(pf), ev_start, ev_len) == (ARG if not_adc else STATE)
            # one rank of one: the boundary record goes to ev_len, the plan made from it to ev_start
            assert L.pp_shard_scan(h, 110.0, -1, ev_len) == want(not_adc), kind
            assert L.pp_shard_plan(h, ev_len, 0, 1, ctypes.byref(p), 0, ev_start) == want(not_adc), kind
            c.sync()
            assert L.pp_shard_commit(h, zeros.ctypes.data_as(_lib._i64p)) == want(not_adc), kind
            assert L.pp_trace_adopt(h, ev_len, 16, 16) == want(not_adc), kind
            put(c, kind, x)                               # adopting made a float32 trace resident
            assert L.pp_trace_prefetch(h, x16.ctypes.data, 16, 0) == want(not_adc), kind
            if not_adc:
                c.swap_trace()
                c.sync()
    finally:
        c.close()
