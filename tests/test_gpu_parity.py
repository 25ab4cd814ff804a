"""GPU parity: the CUDA path (through the C ABI, ctypes) against the CPU oracle and
the reference-generated golden fixtures.

Bars (BASELINE.json north_star): event / segment indices bit-exact; segment
mean/std/min/max within 1e-9 relative (fp64).
"""
import numpy as np
import pytest

import oracle
from conftest import RULES_1000, load_golden
from pypore_b200 import synth

pytestmark = pytest.mark.gpu

STAT_RTOL = 1e-9


def rel_err(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)) if len(a) else 0.0


def gpu_runs(ctx, x32, thr):
    ctx.upload_trace(x32)
    return ctx.runs(ctx.threshold_scan(thr))


def check_runs(ctx, x32, thr):
    got = gpu_runs(ctx, x32, thr)
    want = oracle.threshold_runs(x32.astype(np.float64), thr)
    for g, w, name in zip(got, want, ("start", "length", "min", "max", "below")):
        assert np.array_equal(g, w, equal_nan=True), name
    return got


def gpu_split_f64(ctx, arrays, **kw):
    gain = oracle.min_gain(**kw)
    ctx.upload_events_f64(arrays)
    n = ctx.statsplit(kw.get("min_width", 100), kw.get("max_width", 1000000), kw.get("window_width", 10000), gain)
    ctx.segment_stats()
    return ctx.segments(n)


def check_split_f64(ctx, arrays, **kw):
    # validation mode (every candidate in exact arithmetic) and the production two-stage search
    ctx.set_screening(False)
    ref_tab = gpu_split_f64(ctx, arrays, **kw)
    ctx.set_screening(True)
    tab = gpu_split_f64(ctx, arrays, **kw)
    assert all(np.array_equal(ref_tab[k], tab[k]) for k in ("event", "start", "end"))
    # the barrier-free kernel (k3_flow) against the level-synchronous one (k3_split, the default), both modes
    ctx.set_split_kernel(True)
    try:
        flow = gpu_split_f64(ctx, arrays, **kw)
        ctx.set_screening(False)
        flow_exact = gpu_split_f64(ctx, arrays, **kw)
    finally:
        ctx.set_screening(True)
        ctx.set_split_kernel(False)
    assert all(np.array_equal(flow[k], tab[k]) and np.array_equal(flow_exact[k], tab[k])
               for k in ("event", "start", "end"))
    if max(len(a) for a in arrays) > 10240:
        # long events: the 1024-thread spine kernel (default) against the work-queue CTAs walking the spine
        ctx.set_option(1, 0)
        try:
            alt = gpu_split_f64(ctx, arrays, **kw)
        finally:
            ctx.set_option(1, 1)
        assert all(np.array_equal(alt[k], tab[k]) for k in ("event", "start", "end"))
    k = 0
    for e, a in enumerate(arrays):
        bp = oracle.statsplit(a, **kw)
        edges = np.concatenate(([0], bp, [len(a)]))
        n = len(edges) - 1
        assert np.all(tab["event"][k:k + n] == e)
        assert np.array_equal(tab["start"][k:k + n], edges[:-1]), "event %d starts" % e
        assert np.array_equal(tab["end"][k:k + n], edges[1:]), "event %d ends" % e
        m, s, mn, mx = oracle.segment_stats(a, edges[:-1], edges[1:])
        assert rel_err(tab["mean"][k:k + n], m) < STAT_RTOL
        assert np.max(np.abs(tab["std"][k:k + n] - s)) <= STAT_RTOL * np.max(np.abs(s)) + 1e-300
        assert np.array_equal(tab["min"][k:k + n], mn) and np.array_equal(tab["max"][k:k + n], mx)
        k += n
    assert k == len(tab["start"])
    return tab


# ---------------------------------------------------------------- K1 threshold
def test_threshold_c1_runs_and_events(ctx):
    x = synth.make_trace(60, seed=21, tier="A")
    check_runs(ctx, x, 110.0)
    ne, ns = ctx.select_events(7, 1000, 0, -0.5, 110.0)
    s, l = ctx.events(ne)
    ws, wl = oracle.events(x.astype(np.float64), 110, RULES_1000)
    assert np.array_equal(s, ws) and np.array_equal(l, wl) and ns == wl.sum()
    # default rules (duration > 100000) reject everything here (SURVEY fact 2)
    assert ctx.select_events(7, 100000, 0, -0.5, 110.0)[0] == 0


@pytest.mark.parametrize("n", [1, 2, 3, 5, 31, 32, 33, 4095, 4096, 4097, 8191, 12289, 100003])
def test_threshold_ragged_lengths(ctx, n):
    rng = np.random.RandomState(n)
    x = np.where(rng.uniform(size=n) < 0.5, 50.0, 120.0).astype(np.float32)  # a crossing every ~2 samples
    x += rng.normal(0, 1, n).astype(np.float32)
    check_runs(ctx, x, 110.0)


def test_threshold_edge_cases(ctx):
    # starts and ends below; NaN counts as above and poisons that run's min/max; +-inf
    x = np.array([50, 50, 120, 50, 120, 120, np.nan, 50, 50, np.inf, -np.inf, 50], np.float32)
    got = check_runs(ctx, x, 110.0)
    assert np.isnan(got[2][3]) and np.isnan(got[3][3])
    # no crossing at all, both sides
    check_runs(ctx, np.full(10000, 120.0, np.float32), 110.0)
    check_runs(ctx, np.full(10000, 20.0, np.float32), 110.0)
    # threshold that float32 cannot represent: comparison must be double(x) < thr
    for thr in (110.1, 0.1, -0.3, 1e-50, 3.5e38 * 10):
        xs = np.array([np.float32(thr), np.nextafter(np.float32(thr), np.float32(np.inf)),
                       np.nextafter(np.float32(thr), np.float32(-np.inf)), 0.0, 1e30, -1e30] * 3, np.float32)
        check_runs(ctx, xs, thr)
    # one crossing exactly on every tile boundary and many crossings inside one tile (> 64 local runs)
    x = np.full(4096 * 5 + 17, 120.0, np.float32)
    x[4096:8192] = 30.0
    x[8192 + 100:8192 + 100 + 400:2] = 30.0
    x[-1] = 30.0
    check_runs(ctx, x, 110.0)


def test_threshold_float64_trace(ctx):
    """A float64 trace that float32 cannot hold (int16 counts x a float64 scale, like read_abf.py:208-210) stays
    float64 on the device: runs, extrema, events and the whole pipeline equal the oracle's on the doubles."""
    rng = np.random.RandomState(3)
    x32 = synth.make_trace(12, seed=9, tier="A")
    counts = np.round(x32.astype(np.float64) / 0.0305).astype(np.int16)
    x = counts * 0.0305 + 0.0123                               # read_abf: counts * scale + offset, float64
    assert not np.array_equal(x.astype(np.float32).astype(np.float64), x)
    x[1000:1003] = [np.nan, np.inf, -np.inf]
    thr = 110.0000001                                          # not float32-representable either
    ctx.upload_trace_f64(x)
    got = ctx.runs(ctx.threshold_scan(thr))
    want = oracle.threshold_runs(x, thr)
    for g, w, name in zip(got, want, ("start", "length", "min", "max", "below")):
        assert np.array_equal(g, w, equal_nan=True), name
    x[1000:1003] = x[999]
    ws, wl = oracle.events(x, thr, RULES_1000)
    ctx.upload_trace_f64(x)
    c = ctx.pipeline(thr, rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0,
                     min_width=100, max_width=1000000, window_width=10000,
                     min_gain=oracle.min_gain(prior_segments_per_second=10))
    es, el = ctx.events(c["events"])
    assert np.array_equal(es, ws) and np.array_equal(el, wl) and len(ws) == 12
    oe, ost, oen, _ = oracle.statsplit_events(x, ws, wl, prior_segments_per_second=10)
    t = ctx.segments(c["segments"])
    assert np.array_equal(t["event"], oe) and np.array_equal(t["start"], ost) and np.array_equal(t["end"], oen)
    for e in (0, 5, 11):
        sel = oe == e
        m, s, mn, mx = oracle.segment_stats(x[ws[e]:ws[e] + wl[e]], ost[sel], oen[sel])
        assert rel_err(t["mean"][sel], m) < STAT_RTOL and rel_err(t["std"][sel], s) < STAT_RTOL
        assert np.array_equal(t["min"][sel], mn) and np.array_equal(t["max"][sel], mx)
    # ragged float64 lengths around the tile / span edges
    for n in (1, 5, 511, 512, 513, 4095, 4096, 4097, 8191, 12289):
        y = (np.round(rng.normal(100, 20, n) / 0.0305) * 0.0305)
        ctx.upload_trace_f64(y)
        got = ctx.runs(ctx.threshold_scan(105.0))
        want = oracle.threshold_runs(y, 105.0)
        for g, w, name in zip(got, want, ("start", "length", "min", "max", "below")):
            assert np.array_equal(g, w, equal_nan=True), (n, name)


def test_threshold_dense_crossings_and_span_edges(ctx):
    """More crossings per 512-sample span than k1_scan_tiles stages (the span is walked again by k1_stitch),
    crossings exactly on span / tile boundaries, and NaN inside pieces."""
    rng = np.random.RandomState(11)
    x = rng.normal(100.0, 5.0, 3 * 4096 + 77).astype(np.float32)       # every other sample crosses 100
    check_runs(ctx, x, 100.0)
    y = np.full(5 * 4096, 120.0, np.float32)
    for p in (512, 1024, 4096, 4096 + 511, 8192, 3 * 4096 - 1, 4 * 4096):     # steps exactly at the edges
        y[p:p + 300] = 50.0
    y[515] = np.nan
    y[9000] = np.nan
    check_runs(ctx, y, 110.0)
    z = np.full(4096 * 2, 50.0, np.float32)                             # 9 and 10 crossings in one span, 8 in another
    for k in range(9):
        z[10 + 20 * k] = 120.0 if k % 2 == 0 else 50.0
    z[600:4000:400] = 120.0
    z[4096 + 5:4096 + 5 + 16 * 4:16] = 120.0
    check_runs(ctx, z, 110.0)


def test_threshold_subzero_rule(ctx):
    x = synth.make_trace(40, seed=5, tier="A")
    s, l = oracle.events(x.astype(np.float64), 110, RULES_1000)
    x2, hit = synth.add_subzero_spikes(x, s, l, frac=0.25, seed=3)
    assert len(hit) > 3
    check_runs(ctx, x2, 110.0)
    ne, _ = ctx.select_events(7, 1000, 0, -0.5, 110.0)
    gs, gl = ctx.events(ne)
    ws, wl = oracle.events(x2.astype(np.float64), 110, RULES_1000)
    assert np.array_equal(gs, ws) and np.array_equal(gl, wl) and len(ws) == len(s) - len(hit)


# ---------------------------------------------------------------- K2+K3+K4 split
@pytest.mark.parametrize("kw", [dict(), dict(prior_segments_per_second=10),
                                dict(min_width=50, max_width=2500, window_width=1000, prior_segments_per_second=50),
                                dict(min_width=250, window_width=500),          # window == 2*min_width: never scans
                                dict(min_width=3, max_width=40, window_width=64),
                                dict(min_gain_per_sample=0.01, window_width=2000)])
@pytest.mark.parametrize("tier", ["A", "B"])
def test_split_events_bit_exact(ctx, kw, tier):
    x = synth.make_trace(24, seed=31, tier=tier).astype(np.float64)
    s, l = oracle.events(x, 110, RULES_1000)
    check_split_f64(ctx, [x[a:a + n] for a, n in zip(s, l)], **kw)


def test_split_short_and_degenerate_events(ctx):
    rng = np.random.RandomState(0)
    arrays = [synth.quantise(rng.normal(50, 1, n)).astype(np.float64)
              for n in (1, 2, 7, 199, 200, 201, 202, 399, 400, 401, 1000)]
    arrays.append(np.full(500, 42.0))                       # zero variance: log(0), NaN/inf gains
    arrays.append(np.r_[np.full(300, 42.0), np.full(300, 43.0)])  # +inf gain at the step
    arrays.append(synth.quantise(rng.normal(50, 1, 8000)).astype(np.float64))
    check_split_f64(ctx, arrays)
    check_split_f64(ctx, arrays, min_width=2, max_width=6, window_width=4)   # > K3_LIST items per level
    check_split_f64(ctx, arrays, prior_segments_per_second=10)
    check_split_f64(ctx, arrays, min_width=1, max_width=50, window_width=2)


def test_min_gain_exactly_at_a_decision_boundary(ctx):
    """Windows with one contender are decided from the SCREENED gain when it clears min_gain by more than the
    error bound, and in exact arithmetic otherwise.  Here min_gain is set to gains the reference itself computed
    (and to their floating-point neighbours), so that a decision sits exactly on `gain > min_gain`; the device must
    fall back to exact arithmetic there and reproduce the reference's strict comparison."""
    arrays = [synth.make_long_event(7000, seed=41, tier="A").astype(np.float64),
              synth.make_long_event(5000, seed=42, tier="B").astype(np.float64),
              synth.make_long_event(30000, seed=43, tier="A").astype(np.float64)]   # through the spine kernel
    picked = []
    for a in arrays:
        _, info = oracle.statsplit(a, min_width=100, window_width=10000, return_info=True)
        g = np.sort(info["gains"][np.isfinite(info["gains"])])
        picked += [g[0], g[len(g) // 3], g[len(g) // 2], g[-1]]
    for g in picked:
        for mg in (g, np.nextafter(g, -np.inf), np.nextafter(g, np.inf)):
            ctx.upload_events_f64(arrays)
            n = ctx.statsplit(100, 1000000, 10000, float(mg))
            tab = ctx.segments(n, stats=False)
            k = 0
            for e, a in enumerate(arrays):
                bp = oracle.statsplit(a, min_width=100, window_width=10000, gain=float(mg))
                edges = np.concatenate(([0], bp, [len(a)]))
                m = len(edges) - 1
                assert np.array_equal(tab["start"][k:k + m], edges[:-1]), (g, mg, e)
                assert np.array_equal(tab["end"][k:k + m], edges[1:]), (g, mg, e)
                k += m
            assert k == n


def test_split_long_event_spine_and_forced(ctx):
    """Intervals longer than the shared-memory slab: window chain, queue hand-off, max_width forcing."""
    g = load_golden("long_event.npz")
    x = synth.make_long_event(300000, seed=100, tier="A").astype(np.float64)
    for name, kw in {"long_default": dict(min_width=100, max_width=20000, window_width=10000),
                     "long_psps10": dict(min_width=100, max_width=20000, window_width=10000,
                                         prior_segments_per_second=10),
                     "long_highgain": dict(min_width=100, max_width=15000, window_width=4000,
                                           min_gain_per_sample=2.0)}.items():
        tab = check_split_f64(ctx, [x], **kw)
        assert np.array_equal(tab["start"], g[name + "_start"]) and np.array_equal(tab["end"], g[name + "_end"])
    # window larger than the slab (global-memory scan path), tier B, two long events + short ones
    xb = synth.make_long_event(70000, seed=103, tier="B").astype(np.float64)
    check_split_f64(ctx, [xb, x[:50000], xb[:900]], min_width=100, max_width=1000000, window_width=30000,
                    prior_segments_per_second=10)
    check_split_f64(ctx, [xb], min_width=20, max_width=3000, window_width=14000)


def test_golden_fixture_tables(ctx):
    """Reference-generated tables (tests/golden/make_golden.py) straight against the device pipeline."""
    for name in ("pipeline_tierA.npz", "pipeline_tierB.npz"):
        g = load_golden(name)
        x = synth.make_trace(int(g["n_events"]), seed=int(g["seed"]), tier=str(g["tier"]))
        ctx.upload_trace(x)
        for key, kw in {"default": dict(min_width=100, window_width=10000),
                        "psps10": dict(min_width=100, window_width=10000, prior_segments_per_second=10),
                        "narrow": dict(min_width=50, max_width=2500, window_width=1000,
                                       prior_segments_per_second=50)}.items():
            r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, kw["min_width"], kw.get("max_width", 1000000),
                             kw["window_width"], oracle.min_gain(**kw))
            es, el = ctx.events(r["events"])
            assert np.array_equal(es / float(g["second"]), g["event_start_s"]) and np.array_equal(el, g["event_n"])
            tab = ctx.segments(r["segments"])
            assert np.array_equal(tab["event"], g[key + "_event"])
            assert np.array_equal(tab["start"], g[key + "_start"]) and np.array_equal(tab["end"], g[key + "_end"])
            assert rel_err(tab["mean"], g[key + "_mean"]) < STAT_RTOL
            assert rel_err(tab["std"], g[key + "_std"]) < STAT_RTOL
            assert np.array_equal(tab["min"], g[key + "_min"]) and np.array_equal(tab["max"], g[key + "_max"])
            st = ctx.event_stats(r["events"])
            assert rel_err(st["mean"], g["event_mean"]) < STAT_RTOL and rel_err(st["std"], g["event_std"]) < STAT_RTOL
            assert np.array_equal(st["min"], g["event_min"]) and np.array_equal(st["max"], g["event_max"])


def test_pipeline_c1_full_parity_and_work_counters(ctx):
    """BASELINE config 1 (6 M samples, 500 events), both gain settings, SURVEY known answers."""
    x = synth.make_trace(500, seed=0, tier="A")
    x64 = x.astype(np.float64)
    ctx.upload_trace(x)
    ws, wl = oracle.events(x64, 110, RULES_1000)
    for psps, n_seg in ((None, 30643), (10, 2682)):
        gain = oracle.min_gain(prior_segments_per_second=psps)
        r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain)
        assert (r["runs"], r["events"], r["event_samples"], r["segments"]) == (1001, 500, 3998546, n_seg)
        es, el = ctx.events(r["events"])
        assert np.array_equal(es, ws) and np.array_equal(el, wl)
        tab = ctx.segments(r["segments"])
        oe, ost, oen, ncand = oracle.statsplit_events(x64, ws, wl, gain=gain, threads=8)
        assert np.array_equal(tab["event"], oe) and np.array_equal(tab["start"], ost) and np.array_equal(tab["end"], oen)
        assert ctx.split_counters()["candidates"] == ncand  # same candidate evaluations as the reference
        for e in range(0, 500, 37):
            sel = oe == e
            m, s, mn, mx = oracle.segment_stats(x64[ws[e]:ws[e] + wl[e]], ost[sel], oen[sel])
            assert rel_err(tab["mean"][sel], m) < STAT_RTOL and rel_err(tab["std"][sel], s) < STAT_RTOL
            assert np.array_equal(tab["min"][sel], mn) and np.array_equal(tab["max"][sel], mx)


def test_pipeline_c2_size_properties(ctx):
    """BASELINE config 2 size (60 M samples, 5k events): size-independent properties + sampled oracle parity."""
    x = synth.make_trace(5000, seed=1, tier="A")
    ctx.upload_trace(x)
    mw = 100
    r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, mw, 1000000, 10000, oracle.min_gain())
    assert r["events"] == 5000
    es, el = ctx.events(r["events"])
    tab = ctx.segments(r["segments"])
    # segments partition every event: sorted, contiguous, first starts at 0, last ends at the event length
    assert np.all(np.diff(tab["event"]) >= 0)
    first = np.r_[True, np.diff(tab["event"]) != 0]
    last = np.r_[np.diff(tab["event"]) != 0, True]
    assert np.all(tab["start"][first] == 0) and np.array_equal(tab["end"][last], el)
    assert np.array_equal(tab["start"][~first], tab["end"][:-1][~first[1:]])
    assert np.all(tab["end"] - tab["start"] >= mw)
    # checksum of checksums: sum over segments of n*mean equals the sum of all event samples
    n = (tab["end"] - tab["start"]).astype(np.float64)
    tot = sum(float(x[s:s + l].astype(np.float64).sum()) for s, l in zip(es[::50], el[::50]))
    sel = np.isin(tab["event"], np.arange(0, 5000, 50))
    assert abs(float((n * tab["mean"])[sel].sum()) - tot) <= 1e-9 * abs(tot)
    assert np.all(tab["min"] <= tab["mean"]) and np.all(tab["mean"] <= tab["max"]) and np.all(tab["std"] >= 0)
    # idempotence: same tables on a second pass
    r2 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, mw, 1000000, 10000, oracle.min_gain())
    tab2 = ctx.segments(r2["segments"])
    assert r2 == r and all(np.array_equal(tab[k], tab2[k]) for k in tab)
    # oracle parity on a sample of events
    x64 = x.astype(np.float64)
    for e in range(0, 5000, 250):
        bp = oracle.statsplit(x64[es[e]:es[e] + el[e]])
        sel = tab["event"] == e
        assert np.array_equal(tab["start"][sel][1:], bp)


def test_prefix_modes_agree_and_exactness_proof(ctx):
    """PP_PREFIX_AUTO = tiled scan + exactness proof + sequential redo of unproven events.  ADC-quantised
    data is proven exact (no redo); raw float32 data has inexact sums of squares (every event redone);
    both give the tables of the strict np.cumsum order."""
    from pypore_b200 import _lib
    gain = oracle.min_gain(prior_segments_per_second=10)
    for tier, expect_redo in (("A", 0), ("B", None)):
        x = synth.make_trace(30, seed=77, tier=tier)
        ctx.upload_trace(x)
        ctx.threshold_scan(110.0)
        ne, _ = ctx.select_events(7, 1000, 0, -0.5, 110.0)
        tabs = {}
        for mode in (_lib.PREFIX_SEQUENTIAL, _lib.PREFIX_AUTO):
            n = ctx.statsplit(100, 1000000, 10000, gain, prefix_mode=mode)
            ctx.segment_stats()
            tabs[mode] = ctx.segments(n)
            if mode == _lib.PREFIX_AUTO:
                redo = ctx.split_counters()["seq_redo"]
                assert redo == (ne if expect_redo is None else expect_redo), (tier, redo, ne)
        a, b = tabs[_lib.PREFIX_SEQUENTIAL], tabs[_lib.PREFIX_AUTO]
        assert all(np.array_equal(a[k], b[k]) for k in a)
    # mixed: exact and inexact events in one batch, a long event spanning many tiles, NaN / inf samples
    rng = np.random.RandomState(2)
    arrays = [synth.make_long_event(50000, seed=5, tier="A").astype(np.float64),
              synth.make_long_event(9000, seed=6, tier="B").astype(np.float64),
              synth.quantise(rng.normal(60, 1, 2049)).astype(np.float64),
              rng.normal(60, 1, 2047), np.r_[rng.normal(60, 1, 300), np.nan, rng.normal(60, 1, 300)],
              synth.quantise(rng.normal(60, 1, 1)).astype(np.float64)]
    ctx.upload_events_f64(arrays)
    n = ctx.statsplit(100, 1000000, 10000, gain, prefix_mode=_lib.PREFIX_AUTO)
    assert ctx.split_counters()["seq_redo"] == 3
    check_split_f64(ctx, arrays[:4] + arrays[5:], prior_segments_per_second=10)


def test_screening_error_bound_holds(ctx):
    """The screened value of every valid candidate lies within the eps the kernel assumes of the
    reference-arithmetic value (DESIGN.md derivation), on raw, quantised, filtered-like and low-noise data."""
    rng = np.random.RandomState(5)
    cases = {
        "tierA": synth.make_long_event(40000, seed=7, tier="A").astype(np.float64),
        "tierB": synth.make_long_event(40000, seed=8, tier="B").astype(np.float64),
        "smooth": np.convolve(synth.make_long_event(40100, seed=9, tier="B").astype(np.float64),
                              np.ones(25) / 25, mode="valid")[:40000],          # filtered-like: sigma ~0.2
        "lownoise": 60.0 + 0.02 * rng.normal(size=40000),                         # mean-square / variance ~ 1e7
        "offset": 5000.0 + rng.normal(size=40000),                                # ratio 2.5e7 > 2^24: invalid
        "steps": np.repeat(rng.uniform(20, 90, 40), 1000) + 0.5 * rng.normal(size=40000),
    }
    worst = 0.0
    for name, x in cases.items():
        ctx.upload_events_f64([x])
        ctx.statsplit(100, 1000000, 10000, oracle.min_gain())
        for ps, pe in ((0, 10000), (12345, 22345), (30000, 40000), (100, 700), (20000, 20250)):
            hs, he, ok, eps = ctx.debug_screen(0, ps, pe, 100)
            fin = ok & np.isfinite(he)
            assert np.all(np.isfinite(he[ok])), name                               # valid => exact value finite
            if fin.any():
                err = np.max(np.abs(hs[fin] - he[fin]))
                worst = max(worst, err / eps)
                assert err <= eps, (name, ps, pe, err, eps)
        if name == "offset":
            assert not ok.any()
        if name in ("tierA", "tierB", "steps"):
            assert ok.all()
    assert worst < 0.5      # the bound is conservative
    # production path on the same awkward data stays bit-exact
    check_split_f64(ctx, [cases["lownoise"], cases["offset"][:9000], cases["smooth"][:9000]],
                    prior_segments_per_second=10)
    check_split_f64(ctx, [cases["lownoise"][:9000], cases["steps"][:9500]])


def test_host_selected_events_path(ctx):
    """Arbitrary Python rules: host picks runs from the device run table, pp_set_events feeds the split."""
    x = synth.make_trace(30, seed=8, tier="A")
    x64 = x.astype(np.float64)
    ctx.upload_trace(x)
    runs = ctx.runs(ctx.threshold_scan(110.0))
    keep = np.nonzero(runs[4] & (runs[1] > 7000))[0]  # a rule the device mask cannot express
    ctx.set_events(runs[0][keep], runs[1][keep])
    gain = oracle.min_gain(prior_segments_per_second=10)
    n = ctx.statsplit(100, 1000000, 10000, gain)
    ctx.segment_stats()
    tab = ctx.segments(n)
    oe, ost, oen, _ = oracle.statsplit_events(x64, runs[0][keep], runs[1][keep], gain=gain)
    assert np.array_equal(tab["event"], oe) and np.array_equal(tab["start"], ost) and np.array_equal(tab["end"], oen)


# ---------------------------------------------------------------- K5 filter
FILTER_RTOL = 1e-5   # BASELINE.json north_star: filtered current within 1e-5 relative


@pytest.mark.parametrize("name", ["filter_o1_100k.npz", "filter_o1_250k.npz", "filter_o2_100k.npz",
                                  "filter_o4_100k.npz"])
def test_filter_matches_scipy_fixture(ctx, name):
    """Event.filter arithmetic against what the reference (scipy.signal.filtfilt) produced."""
    from pypore_b200.DataTypes import bessel_coefficients
    g = load_golden(name)
    x = synth.make_trace(3, seed=int(g["seed"]), tier="A").astype(np.float64)
    start, length = oracle.events(x, 110, RULES_1000)
    b, a, zi = bessel_coefficients(int(g["order"]), float(g["cutoff"]), float(g["fs"]))
    evs = [x[start[i]:start[i] + length[i]] for i in range(2)]
    ctx.upload_events_f64(evs)
    ctx.filter_events(b, a, zi)
    y = ctx.event_samples(int(length[:2].sum()))
    ref = np.concatenate([g["event0_filtered"], g["event1_filtered"]])
    err = np.max(np.abs(y - ref) / np.abs(ref))
    assert err < FILTER_RTOL, err
    assert err < 1e-10          # in practice the scan agrees with scipy to rounding
    # segmentation of the filtered events (float64 path) equals the reference's on its own filtered signal
    kw = dict(min_width=100, window_width=10000, sampling_freq=float(g["fs"]), cutoff_freq=float(g["cutoff"]),
              prior_segments_per_second=10)
    n = ctx.statsplit(100, 1000000, 10000, oracle.min_gain(**kw))
    ctx.segment_stats()
    tab = ctx.segments(n)
    for i in range(2):
        sel = tab["event"] == i
        assert np.array_equal(tab["start"][sel], g["event%d_seg_start" % i])
        assert np.array_equal(tab["end"][sel], g["event%d_seg_end" % i])
        assert rel_err(tab["mean"][sel], g["event%d_seg_mean" % i]) < 1e-9
        assert rel_err(tab["std"][sel], g["event%d_seg_std" % i]) < 1e-7   # std of a 1e-15-perturbed signal


def test_filter_edge_lengths_and_orders(ctx):
    from pypore_b200.DataTypes import bessel_coefficients
    rng = np.random.RandomState(3)
    for order, fs in ((1, 1e5), (2, 1e5), (3, 2.5e5), (4, 1e5), (6, 1e5), (8, 1e5)):
        b, a, zi = bessel_coefficients(order, 2000., fs)
        pad = 3 * (order + 1)
        lens = [pad + 1, pad + 2, 100, 4095, 4096 - 2 * pad, 4097, 8192, 20011]
        evs = [60 + rng.normal(0, 2, n) for n in lens]
        ctx.upload_events_f64(evs)
        ctx.filter_events(b, a, zi)
        y = ctx.event_samples(sum(lens))
        k = 0
        for e in evs:
            ref = oracle.filtfilt(b, a, e)
            got = y[k:k + len(e)]
            err = np.max(np.abs(got - ref) / np.abs(ref))
            assert err < FILTER_RTOL, (order, len(e), err)
            # orders 1-2: parallel scan (rounding differs from the sequential order, measured <= 2e-9);
            # orders 3-8: scipy's own operation order, bit-identical to the oracle
            assert err < (1e-8 if order <= 3 else 1e-15), (order, len(e), err)
            k += len(e)
        # not longer than padlen: scipy raises ValueError
        ctx.upload_events_f64([evs[2], evs[0][:pad]])
        with pytest.raises(ValueError, match="padlen"):
            ctx.filter_events(b, a, zi)


def test_filtered_pipeline_on_float32_trace(ctx):
    """BASELINE config 5 shape: threshold -> Event.filter(1, 2000) -> SpeedyStatSplit, device resident."""
    from pypore_b200.DataTypes import bessel_coefficients
    fs = 2.5e5
    x = synth.make_trace(40, seed=1000, tier="A")
    x64 = x.astype(np.float64)
    ctx.upload_trace(x)
    b, a, zi = bessel_coefficients(1, 2000., fs)
    kw = dict(min_width=100, window_width=10000, sampling_freq=fs, cutoff_freq=2000., prior_segments_per_second=10)
    r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, oracle.min_gain(**kw),
                     filter_ba=(b, a, zi))
    ws, wl = oracle.events(x64, 110, RULES_1000)
    es, el = ctx.events(r["events"])
    assert np.array_equal(es, ws) and np.array_equal(el, wl)
    y = ctx.event_samples(r["event_samples"])
    tab = ctx.segments(r["segments"])
    off = np.concatenate(([0], np.cumsum(wl)))
    flips = 0
    for e in range(len(ws)):
        ref = oracle.filtfilt(b, a, x64[ws[e]:ws[e] + wl[e]])
        got = y[off[e]:off[e + 1]]
        assert np.max(np.abs(got - ref) / np.abs(ref)) < FILTER_RTOL
        sel = tab["event"] == e
        # bit-exact against the oracle run on the very samples the device segmented
        assert np.array_equal(tab["start"][sel][1:], oracle.statsplit(got, **kw))
        m, s, mn, mx = oracle.segment_stats(got, tab["start"][sel], tab["end"][sel])
        assert rel_err(tab["mean"][sel], m) < STAT_RTOL and rel_err(tab["std"][sel], s) < STAT_RTOL
        assert np.array_equal(tab["min"][sel], mn) and np.array_equal(tab["max"][sel], mx)
        flips += not np.array_equal(tab["start"][sel][1:], oracle.statsplit(ref, **kw))
    assert flips == 0   # and the scipy-filtered signal segments identically on this suite


def test_hardware_lg2_error_within_screening_bound(ctx):
    """Exhaustive over all 2^23 mantissas: the 23-bit fixed-point log2 built from MUFU.LG2 plus one float32
    addition stays within the 2^-22 + 2^-24 the screening bound (split.cuh K3_EPS_PER_SAMPLE) assumes."""
    err = ctx.debug_lg2_error()
    assert 0.0 < err <= 2.0 ** -22 + 2.0 ** -24, err


@pytest.mark.parametrize("chunk", [4096, 65536, 1 << 20])
def test_streamed_host_pipeline_equals_resident(ctx, chunk):
    """pp_pipeline_host (chunked copy overlapped with scan / select / prefix / split per chunk) returns exactly
    the tables of upload + pp_pipeline, for chunk sizes that cut events, gaps and K1 tiles in every way;
    the trace starts and ends below the threshold so that the open first/last runs are events too."""
    body = synth.make_trace(60, seed=21, tier="A")
    lead = synth.quantise(np.random.RandomState(3).normal(50, 1, 5000)).astype(np.float32)
    x = np.concatenate([lead, body, lead[:3000]])
    x64 = x.astype(np.float64)
    for psps in (None, 10):
        gain = oracle.min_gain(prior_segments_per_second=psps)
        ctx.upload_trace(x)
        r0 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain)
        ev0, tab0, c0 = ctx.events(r0["events"]), ctx.segments(r0["segments"]), ctx.split_counters()
        r1 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain, host_trace=x,
                          chunk_samples=chunk)
        ev1, tab1, c1 = ctx.events(r1["events"]), ctx.segments(r1["segments"]), ctx.split_counters()
        assert r1 == r0 and r0["events"] == 62
        assert np.array_equal(ev0[0], ev1[0]) and np.array_equal(ev0[1], ev1[1])
        assert all(np.array_equal(tab0[k], tab1[k]) for k in tab0)
        assert c1["candidates"] == c0["candidates"] and c1["scans"] == c0["scans"]
        ws, wl = oracle.events(x64, 110, RULES_1000)
        assert np.array_equal(ev1[0], ws) and np.array_equal(ev1[1], wl)
        oe, ost, oen, _ = oracle.statsplit_events(x64, ws, wl, gain=gain)
        assert np.array_equal(tab1["event"], oe) and np.array_equal(tab1["start"], ost) and np.array_equal(tab1["end"], oen)
        # pp_pipeline_host_tables: compaction / statistics / copy-out per chunk into page-locked host tables
        r2 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain, host_trace=x,
                          chunk_samples=chunk, export=True)
        assert {k: r2[k] for k in r0} == r0
        assert np.array_equal(r2["event_table"][0], ev0[0]) and np.array_equal(r2["event_table"][1], ev0[1])
        assert set(r2["segment_table"]) == set(tab0)
        assert all(np.array_equal(tab0[k], r2["segment_table"][k]) for k in tab0)
        # ... and the device tables it leaves behind are the same ones
        tab2 = ctx.segments(r2["segments"])
        assert all(np.array_equal(tab0[k], tab2[k]) for k in tab0)


def test_host_tables_too_small_fall_back_to_downloads(ctx):
    """More events than the exporting call reserves host rows for: the C call reports PP_ERR_CAPACITY, the Python
    layer fetches the (complete) device tables instead."""
    n = 1200000
    x = np.where((np.arange(n) // 50) % 2 == 0, 50.0, 120.0).astype(np.float32)   # 12,000 events of 50 samples
    x += (np.arange(n) % 7).astype(np.float32) * 0.125
    gain = oracle.min_gain()
    kw = dict(host_trace=x, chunk_samples=1 << 18)
    r = ctx.pipeline(110.0, 5, 20, 0, 0.0, 110.0, 10, 1000000, 40, gain, export=True, **kw)
    assert r["events"] == 12000 and r["events"] > n // 256 + 4096
    ctx.upload_trace(x)
    r0 = ctx.pipeline(110.0, 5, 20, 0, 0.0, 110.0, 10, 1000000, 40, gain)
    tab0 = ctx.segments(r0["segments"])
    assert {k: r[k] for k in r0} == r0
    assert all(np.array_equal(tab0[k], r["segment_table"][k]) for k in tab0)


def test_streamed_host_pipeline_no_events_and_single_chunk(ctx):
    rng = np.random.RandomState(4)
    x = synth.quantise(rng.normal(120, 1.5, 300000)).astype(np.float32)   # never below the threshold
    r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, oracle.min_gain(), host_trace=x,
                     chunk_samples=8192)
    assert (r["runs"], r["events"], r["segments"]) == (1, 0, 0)
    x = synth.make_trace(5, seed=2, tier="A")                               # shorter than one chunk
    r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, oracle.min_gain(), host_trace=x)
    r2 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, oracle.min_gain(), host_trace=x,
                      export=True)
    ctx.upload_trace(x)
    r0 = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, oracle.min_gain())
    assert r == r0 and {k: r2[k] for k in r0} == r0
    tab0 = ctx.segments(r0["segments"])
    assert all(np.array_equal(tab0[k], r2["segment_table"][k]) for k in tab0)


def test_pinned_downloads_and_pinned_trace(ctx):
    """Page-locked host buffers: a pinned trace through the streamed pipeline and the pinned segment table
    equal the pageable path."""
    x = synth.make_trace(20, seed=5, tier="A")
    xp = ctx.pinned_empty(len(x), np.float32)
    xp[:] = x
    gain = oracle.min_gain(prior_segments_per_second=10)
    r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain, host_trace=xp, chunk_samples=65536)
    a = ctx.segments(r["segments"])
    b = ctx.segments(r["segments"], pinned=True)
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    c = ctx.segments(r["segments"], stats=False, pinned=True)
    assert set(c) == {"event", "start", "end"} and np.array_equal(c["end"], a["end"])


def test_prefetched_traces_queue_two_deep(ctx):
    """pp_trace_prefetch / pp_trace_swap: two traces may be on their way while the resident one is processed; they
    become resident oldest first, each gives exactly the tables of a plain upload, a third prefetch is refused."""
    import torch
    from pypore_b200 import _lib
    gain = oracle.min_gain()
    traces = [synth.make_trace(n, seed=s, tier="A") for n, s in ((12, 41), (20, 42), (7, 43), (15, 44))]
    want = []
    for x in traces:
        ctx.upload_trace(x)
        r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain)
        want.append((r, ctx.events(r["events"]), ctx.segments(r["segments"])))
    pinned = [torch.from_numpy(x).pin_memory().numpy() for x in traces]
    ctx.upload_trace(pinned[0])
    ctx.prefetch_trace(pinned[1])
    ctx.prefetch_trace(pinned[2], extra_capacity=1000)
    with pytest.raises(_lib.PyPoreCudaError):
        ctx.prefetch_trace(pinned[3])
    for k in range(4):
        r = ctx.pipeline(110.0, 7, 1000, 0, -0.5, 110.0, 100, 1000000, 10000, gain)
        ev, tab = ctx.events(r["events"]), ctx.segments(r["segments"])
        assert r == want[k][0], k
        assert np.array_equal(ev[0], want[k][1][0]) and np.array_equal(ev[1], want[k][1][1])
        assert all(np.array_equal(tab[c], want[k][2][c], equal_nan=True) for c in tab)
        if k == 1:
            ctx.prefetch_trace(pinned[3])       # the queue refills while it drains
        if k < 3:
            ctx.swap_trace()
            assert ctx.prefetch_ms() > 0.0
    with pytest.raises(_lib.PyPoreCudaError):
        ctx.swap_trace()                        # nothing left
