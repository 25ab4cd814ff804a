"""int16 ADC traces on the device: every result equals the oracle's on the float64 current decode(counts) and the
existing float32 / float64 paths' on the same values."""
import ctypes

import numpy as np
import pytest

import oracle
from conftest import RULES_1000
from pypore_b200 import _lib, synth
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import File
from pypore_b200.parsers import RuleSet, SpeedyStatSplit, lambda_event_parser, statsplit_min_gain

pytestmark = pytest.mark.gpu

RULES = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
REAL = (0.0305, 0.0123)    # a non-dyadic scale: the decoded current is not float32-representable


def adc_of(x32, scale=1.0 / 32, offset=0.0):
    return AdcTrace(np.round((x32.astype(np.float64) - offset) / scale).astype(np.int16), scale, offset)


def check_runs(ctx, t, thr):
    ctx.upload_trace_adc16(t)
    got = ctx.runs(ctx.threshold_scan(thr))
    want = oracle.threshold_runs(t.decode(), thr)
    for g, w, name in zip(got, want, ("start", "length", "min", "max", "below")):
        assert np.array_equal(g, w, equal_nan=True), (len(t), t.scale, thr, name)
        if g.dtype == np.float64:
            assert g.tobytes() == w.tobytes(), name      # bitwise, signed zeros included


def gains():
    return statsplit_min_gain(**SPLIT)[3]


def tables(ctx, r):
    es, el = ctx.events(r["events"])
    return (es, el), ctx.segments(r["segments"])


def assert_same_tables(a, b, rtol):
    (ea, la), sa = a
    (eb, lb), sb = b
    assert np.array_equal(ea, eb) and np.array_equal(la, lb)
    for k in ("event", "start", "end"):
        assert np.array_equal(np.asarray(sa[k], np.int64), np.asarray(sb[k], np.int64)), k
    for k in ("mean", "std"):
        assert np.allclose(sa[k], sb[k], rtol=rtol, atol=0), k
    for k in ("min", "max"):
        assert np.array_equal(sa[k], sb[k]), k


def test_runs_threshold_edge_cases_both_signs(ctx):
    rng = np.random.RandomState(1)
    c = rng.randint(-400, 400, 3 * 4096 + 77).astype(np.int16)
    c[100:110] = (-32768, 32767, -32768, 32767, 0, 0, -1, 1, -32768, 32767)
    for scale, offset in ((0.0305, 0.0123), (-0.0305, 0.0123), (1.0 / 32, 0.0), (-1.0 / 32, -0.0), (0.25, -0.0)):
        t = AdcTrace(c, scale, offset)
        vals = np.unique(t.decode())
        for thr in (vals[len(vals) // 2], (vals[10] + vals[11]) / 2, vals[0] - 1, vals[-1] + 1, vals[0], vals[-1],
                    np.nan, np.inf, -np.inf, 0.0):
            check_runs(ctx, t, thr)


def test_runs_ragged_lengths_and_dense_crossings(ctx):
    rng = np.random.RandomState(2)
    for n in (1, 2, 5, 511, 512, 513, 4095, 4096, 4097, 8191, 12289, 100003):
        for scale in (0.0305, -0.0305):
            t = AdcTrace((rng.normal(0, 40, n)).astype(np.int16), scale, 0.0123)
            check_runs(ctx, t, 0.0)
    t = AdcTrace(np.full(5 * 4096, 100, np.int16), 1.0 / 32)        # no crossing, both sides
    check_runs(ctx, t, 1.0)
    check_runs(ctx, t, 10.0)
    c = np.full(5 * 4096 + 17, 3000, np.int16)
    c[4096:8192] = 100                                            # crossings on tile boundaries
    c[8192 + 100:8192 + 500:2] = 100                              # more crossings per span than are staged
    check_runs(ctx, AdcTrace(c, 0.0305, 0.0123), 50.0)
    check_runs(ctx, AdcTrace(c, -0.0305, 0.0123), -50.0)


def test_tier_a_adc_equals_float32_path(ctx):
    x = synth.make_trace(60, seed=21, tier="A")
    t = adc_of(x)
    assert np.array_equal(t.decode(), x.astype(np.float64))
    ctx.upload_trace(x)
    want = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), **SPLIT, **RULES))
    c_want = ctx.split_counters()
    ctx.upload_trace_adc16(t)
    got = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), **SPLIT, **RULES))
    assert_same_tables(got, want, 1e-12)
    c_got = ctx.split_counters()
    for k in ("candidates", "scans", "tasks", "exact"):
        assert c_got[k] == c_want[k], k
    assert len(got[0][0]) == 60


def test_non_dyadic_scale_equals_float64_trace_path(ctx):
    x = synth.make_trace(40, seed=22, tier="A")
    t = adc_of(x, *REAL)
    x64 = t.decode()
    assert not np.array_equal(x64.astype(np.float32).astype(np.float64), x64)
    for mode in (_lib.PREFIX_AUTO, _lib.PREFIX_SEQUENTIAL):
        ctx.upload_trace_f64(x64)
        want = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), prefix_mode=mode, **SPLIT, **RULES))
        c_want = ctx.split_counters()
        ctx.upload_trace_adc16(t)
        got = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), prefix_mode=mode, **SPLIT, **RULES))
        assert_same_tables(got, want, 1e-9)
        assert ctx.split_counters() == c_want           # candidates, scans, strict-order redos (n_seq_redo), ...
        if mode == _lib.PREFIX_AUTO:
            assert c_want["seq_redo"] > 0               # a non-dyadic current does need the strict-order redo
    # and the oracle on the decoded current
    ws, wl = oracle.events(x64, 110.0, RULES_1000)
    assert np.array_equal(got[0][0], ws) and np.array_equal(got[0][1], wl)
    oe, ost, oen, _ = oracle.statsplit_events(x64, ws, wl)
    assert np.array_equal(got[1]["event"], oe) and np.array_equal(got[1]["start"], ost)
    for e in (0, 17, 39):
        sel = oe == e
        m, s, mn, mx = oracle.segment_stats(x64[ws[e]:ws[e] + wl[e]], ost[sel], oen[sel])
        assert np.allclose(got[1]["mean"][sel], m, rtol=1e-9, atol=0)
        assert np.allclose(got[1]["std"][sel], s, rtol=1e-9, atol=0)
        assert np.array_equal(got[1]["min"][sel], mn) and np.array_equal(got[1]["max"][sel], mx)
    # per-event statistics, prefix sums and exact window gains on the resident ADC trace
    ctx.upload_trace_adc16(t)
    ctx.threshold_scan(110.0)
    ne, _ = ctx.select_events(**RULES)
    ev_adc = ctx.event_stats(ne)
    ctx.prefix()
    g_adc = ctx.window_gains(3, [0, 500], [3000, 5000], 100)
    ctx.upload_trace_f64(x64)
    ctx.threshold_scan(110.0)
    ctx.select_events(**RULES)
    ev_64 = ctx.event_stats(ne)
    ctx.prefix()
    g_64 = ctx.window_gains(3, [0, 500], [3000, 5000], 100)
    for k in ("min", "max"):
        assert np.array_equal(ev_adc[k], ev_64[k])
    for k in ("mean", "std"):
        assert np.allclose(ev_adc[k], ev_64[k], rtol=1e-9, atol=0)
    assert all(np.array_equal(a, b) for a, b in zip(g_adc, g_64))


def test_negative_scale_pipeline(ctx):
    x = synth.make_trace(12, seed=23, tier="A")
    t = AdcTrace(np.round(-x.astype(np.float64) / 0.0305).astype(np.int16), -0.0305, 0.0123)
    ctx.upload_trace_f64(t.decode())
    want = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), **SPLIT, **RULES))
    ctx.upload_trace_adc16(t)
    got = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), **SPLIT, **RULES))
    assert_same_tables(got, want, 1e-9)
    assert len(got[0][0]) == 12


def test_file_parse_filtered_250khz_equals_float64_path():
    x = synth.make_trace(10, seed=24, tier="A")
    t = adc_of(x, *REAL)
    seg = SpeedyStatSplit(min_width=100, window_width=10000, sampling_freq=2.5e5, cutoff_freq=2000.,
                          prior_segments_per_second=10)
    det = lambda_event_parser(threshold=110, rules=RuleSet(duration_gt=1000, min_gt=-0.5, max_lt=110))
    out = []
    for cur in (t, t.decode()):
        f = File(current=cur, timestep=1000. / 2.5e5)
        f.parse(parser=det, segmenter=seg, filter_params=(1, 2000))
        out.append(f)
    a, b = out
    assert "current" not in a.__dict__                            # the parse never decoded the whole trace
    for k in ("start", "length", "min", "max"):
        assert np.array_equal(a.event_table[k], b.event_table[k]), k
    for k in ("event", "start", "end", "min", "max"):
        assert np.array_equal(a.segment_table[k], b.segment_table[k]), k
    for k in ("mean", "std"):
        assert np.allclose(a.segment_table[k], b.segment_table[k], rtol=1e-9, atol=0)
    assert len(a.events) == 10
    ea, eb = a.events[4], b.events[4]
    assert np.array_equal(ea.current, eb.current) and ea.filtered
    assert np.array_equal(ea.segments[2].current, eb.segments[2].current)
    # unfiltered, with a segmenter and with none
    for kw in (dict(segmenter=seg), dict()):
        fa, fb = File(current=t, timestep=0.01), File(current=t.decode(), timestep=0.01)
        fa.parse(parser=det, **kw)
        fb.parse(parser=det, **kw)
        for k in ("start", "length", "min", "max"):
            assert np.array_equal(fa.event_table[k], fb.event_table[k]), k
        assert fa.events[3].current.tobytes() == fb.events[3].current.tobytes()


@pytest.mark.parametrize("export", [False, True])
def test_streamed_host_pipeline_equals_resident(ctx, export):
    x = synth.make_trace(80, seed=25, tier="A")
    for scale, offset in ((1.0 / 32, 0.0), REAL):
        t = adc_of(x, scale, offset)
        ctx.upload_trace_adc16(t)
        want = tables(ctx, ctx.pipeline(110.0, min_gain=gains(), **SPLIT, **RULES))
        c_want = ctx.split_counters()
        counts = ctx.pinned_empty(len(t), np.int16)
        counts[:] = t.counts
        pinned = AdcTrace(counts, scale, offset)
        for chunk in (4096 * 5, 4096 * 37 + 1, 100000, 0):
            r = ctx.pipeline(110.0, min_gain=gains(), host_trace=pinned, chunk_samples=chunk, export=export,
                             **SPLIT, **RULES)
            if export:
                es, el = r["event_table"]
                got = ((np.asarray(es), np.asarray(el)), r["segment_table"])
            else:
                got = tables(ctx, r)
            assert_same_tables(got, want, 1e-12)
            assert ctx.split_counters()["candidates"] == c_want["candidates"]
            assert ctx.split_counters()["seq_redo"] == c_want["seq_redo"]


def test_host_evaluated_python_rules():
    x = synth.make_trace(8, seed=26, tier="A")
    t = adc_of(x, *REAL)
    rules = [lambda e: e.duration > 1000, lambda e: e.min > -0.5, lambda e: np.mean(e.current) < 100.0]
    a = lambda_event_parser(threshold=110, rules=rules).parse(t)
    b = lambda_event_parser(threshold=110, rules=rules).parse(t.decode())
    assert len(a) == len(b) > 0
    for sa, sb in zip(a, b):
        assert sa.start == sb.start and sa.duration == sb.duration
        assert sa.current.dtype == np.float64 and sa.current.tobytes() == sb.current.tobytes()


def test_empty_and_one_sample_traces(ctx):
    empty = AdcTrace(np.zeros(0, np.int16), 0.0305)
    f = File(current=empty, timestep=0.01)
    f.parse(parser=lambda_event_parser(threshold=110, rules=RuleSet(duration_gt=1000, min_gt=-0.5, max_lt=110)),
            segmenter=SpeedyStatSplit(min_width=100, window_width=10000))
    assert len(f.events) == 0
    assert lambda_event_parser(threshold=110).parse(empty) == []
    for c in (-32768, 0, 32767):
        check_runs(ctx, AdcTrace(np.array([c], np.int16), 0.0305, 0.0123), 0.0)


def test_float32_only_calls_refuse_an_adc_trace(ctx):
    L = _lib.load()
    t = adc_of(synth.make_trace(2, seed=27, tier="A"))
    ctx.upload_trace_adc16(t)
    h = ctx._h
    x32 = np.zeros(16, np.float32)
    rec = np.zeros(16, np.int64)
    p, _ = ctx._params(110.0, min_width=100, max_width=1000000, window_width=10000, min_gain=0.0, **RULES)
    assert L.pp_trace_append(h, x32.ctypes.data, 16, 0) == _lib.PP_ERR_STATE
    assert L.pp_trace_extend(h, 0) == _lib.PP_ERR_STATE
    assert L.pp_trace_prefetch(h, x32.ctypes.data, 16, 0) == _lib.PP_ERR_STATE
    assert L.pp_trace_adopt(h, ctx.table_ptr(7), 16, 16) == _lib.PP_ERR_STATE
    assert L.pp_shard_scan(h, 110.0, -1, ctypes.c_void_p(ctx.table_ptr(7))) == _lib.PP_ERR_STATE
    assert L.pp_shard_finish(h, ctypes.byref(p), 0, 0, 0, 0, 0, ctypes.c_void_p(ctx.table_ptr(7))) == _lib.PP_ERR_STATE
    assert L.pp_shard_commit(h, rec.ctypes.data_as(_lib._i64p)) == _lib.PP_ERR_STATE
    # invalid decodings are refused by the C entry points too
    assert L.pp_trace_upload_adc16(h, t.counts.ctypes.data, len(t), 0.0, 0.0) == _lib.PP_ERR_ARG
    out = np.zeros(4, np.int64)
    assert L.pp_pipeline_host_adc16(h, t.counts.ctypes.data, len(t), np.nan, 0.0, 0, ctypes.byref(p), None,
                                    out.ctypes.data_as(_lib._i64p)) == _lib.PP_ERR_ARG
    # the context still works, and a float32 trace takes the float32 calls again
    ctx.upload_trace(x32 + 120.0)
    assert L.pp_trace_extend(h, 0) == _lib.PP_OK
