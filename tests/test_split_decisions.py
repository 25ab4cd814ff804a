"""The split search's window decisions (K3) against the reference rule, case by case.

Each case family is built so that a window decision takes a branch the synthetic traces almost never reach: exact
ties, several +inf gains, NaN gains, non-finite and extreme samples, windows with hundreds of contenders within the
screening bound, levels with dozens of short windows.  The device is compared with the reference's rule
(first occurrence of the largest gain above min_gain, strict '>', NaN never wins, cparsers.pyx:149-151).

The oracle evaluates `log` with glibc, the device with CUDA; the two may differ by an ulp or so, which moves a gain
by up to ~3e-10 (tests/test_margin_audit.py).  A decision closer than that has no defined answer, so the CPU test
test_every_decision_is_robust checks, for every window scan of every case, that the decision is one of
  * clear by at least REQUIRED: best minus runner-up, and best against min_gain;
  * decided by +-inf or NaN gains, which no rounding of `log` can change;
  * an exact tie whose operands are identical: the tied candidates' {(n1, V1), (n2, V2)} are bitwise equal as
    multisets, V restated with the reference's own operations, so any `log` gives equal gains;
and that each case reaches the branch its name promises.
"""
from fractions import Fraction

import numpy as np
import pytest

import oracle

REQUIRED = 3e-9
U = 2.0 ** -53


def q32(a):
    return np.round(np.asarray(a, np.float64) * 32.0) / 32.0


def rng(seed):
    return np.random.RandomState(seed)


# ---------------------------------------------------------------------------------------------- case families
def mirror(half):
    return np.concatenate([half, half[::-1]])


def _levels(r, sizes, levels, sd):
    return np.concatenate([q32(lv + r.normal(0, sd, n)) for n, lv in zip(sizes, levels)])


def case_mirror_short():
    r = rng(1)
    arrays = [mirror(_levels(r, (a, b), (100.0, 80.0), 1.0)) for a, b in ((150, 250), (120, 180), (260, 90))]
    return dict(arrays=arrays, kw=dict(min_width=50, window_width=2000, prior_segments_per_second=10))


def case_mirror_far():
    """One window of 4000 samples; the tied pair sits in opposite halves, in different warps' pieces."""
    r = rng(2)
    arrays = [mirror(_levels(r, (1000, 1000), (100.0, 70.0), 1.0))]
    return dict(arrays=arrays, kw=dict(min_width=100, window_width=4000, prior_segments_per_second=10))


def case_mirror_spine():
    """An event longer than one CTA resolves: its first window (palindromic) is scanned by the spine cluster, the
    tied candidates in different CTAs of it."""
    r = rng(3)
    head = mirror(_levels(r, (1400, 2696), (100.0, 75.0), 1.0))
    tail = _levels(r, (3000, 4000, 2500, 3000, 3500), (90.0, 60.0, 95.0, 70.0, 85.0), 1.0)
    return dict(arrays=[np.concatenate([head, tail])],
                kw=dict(min_width=100, window_width=8192, prior_segments_per_second=10))


def case_inf_gains():
    r = rng(4)
    noise = lambda n, lv=100.0: q32(lv + r.normal(0, 1, n))
    arrays = [np.r_[np.full(300, 42.0), noise(700)],               # +inf for every candidate with a constant left side
              np.r_[noise(600), np.full(400, 42.0)],               # ... constant right side
              np.r_[np.full(150, 42.0), np.full(350, 43.0)],       # both sides: all +inf, the first wins
              np.full(500, 42.0),                                  # tot = -inf, every gain NaN, no split
              np.r_[np.full(100, 42.0), noise(500)],               # constant run ending exactly at ps + mw
              np.r_[noise(500), np.full(100, 42.0)],               # ... starting exactly at pe - mw
              np.r_[noise(300), np.full(5000, 7.0)]]               # constant tail longer than a window
    return dict(arrays=arrays, kw=dict(min_width=100, window_width=1000))


def _nonfinite_rows():
    r = rng(5)
    base = lambda: _levels(r, (300, 300, 400), (100.0, 70.0, 90.0), 1.0)
    rows = []
    for v in (np.nan, np.inf, -np.inf):
        for pos in (0, 500, 999):
            a = base()
            a[pos] = v
            rows.append(a)
    z = np.where(r.uniform(size=600) < 0.5, -0.0, 0.0)
    rows.append(np.r_[z, q32(5.0 + r.normal(0, 1, 400))])          # mixed -0.0 / +0.0
    return rows


def case_nonfinite():
    return dict(arrays=_nonfinite_rows(), kw=dict(min_width=50, window_width=1000, prior_segments_per_second=10))


def case_extreme():
    """x*x overflows (1e155) or is subnormal / 0 (1e-160): representable in float64 only."""
    r = rng(6)
    big = _levels(r, (300, 300, 400), (100.0, 70.0, 90.0), 1.0) * 2.0 ** 512
    tiny = _levels(r, (300, 300, 400), (100.0, 70.0, 90.0), 1.0) * 2.0 ** -540
    mixed = np.r_[_levels(r, (400,), (100.0,), 1.0), tiny[:300], _levels(r, (300,), (80.0,), 1.0)]
    return dict(arrays=[big, tiny, mixed], kw=dict(min_width=50, window_width=1000, prior_segments_per_second=10))


def case_crowded():
    """x = +-1 alternating: every candidate of the window is within 2 eps of the best (several hundred contenders,
    more than the exact-evaluation requests a level holds); the two ends tie exactly."""
    n = 4096
    x = np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
    return dict(arrays=[x, x[:3000].copy()], kw=dict(min_width=1001, window_width=4096))


def case_full_levels():
    """Levels wider than the 128 windows a CTA lists: a staircase of 1024 four-sample steps resolves into a bushy
    tree of short windows while the interval behind it walks a quiet stretch window by window (ps > s).  The quiet
    windows fail the validity test (mean^2 / variance > 2^24), so they are scanned exactly after every other window
    of their level has registered its children: the advanced interval is registered past the list and goes to the
    global queue."""
    arrays = []
    for seed in (1, 2, 3):
        r = rng(seed)
        busy = np.repeat(4.0 * np.arange(1024), 4) + q32(r.normal(0, 0.25, 4096))
        arrays.append(np.r_[busy, q32(5000.0 + r.normal(0, 0.25, 6000))])
    return dict(arrays=arrays, kw=dict(min_width=2, window_width=2048, prior_segments_per_second=10))


def case_validity():
    """The screen's validity test at its edges: DC offsets that put (S/n)^2 / V below, around and above 2^24; a
    quiet stretch (sigma ~ 1e-20) next to a loud one (sigma ~ 1e20), so that candidate variances leave ebase +- 127;
    windows whose own variance k3_window_ebase rejects (too small, too large)."""
    r = rng(9)
    arrays = []
    for dc in (2048.0, 4096.0, 8192.0):
        arrays.append(_levels(r, (400, 400), (dc, dc + 40.0), 1.0))
    quiet = q32(r.normal(0, 1, 400)) * 2.0 ** -66
    loud = q32(r.normal(0, 1, 400)) * 2.0 ** 66
    arrays.append(np.r_[quiet, loud])
    arrays.append(np.r_[quiet, loud, quiet])
    arrays.append(_levels(r, (400, 400), (100.0, 60.0), 1.0) * 2.0 ** -470)
    arrays.append(_levels(r, (400, 400), (100.0, 60.0), 1.0) * 2.0 ** 450)
    return dict(arrays=arrays, kw=dict(min_width=50, window_width=1000, prior_segments_per_second=10))


CASES = {
    "mirror_short": case_mirror_short,
    "mirror_far": case_mirror_far,
    "mirror_spine": case_mirror_spine,
    "inf_gains": case_inf_gains,
    "nonfinite": case_nonfinite,
    "extreme": case_extreme,
    "crowded": case_crowded,
    "full_levels": case_full_levels,
    "validity": case_validity,
}


def split_kw(kw):
    kw = dict(kw)
    gain = kw.pop("gain", None)
    mw, MW, W = kw.pop("min_width", 100), kw.pop("max_width", 1000000), kw.pop("window_width", 10000)
    if gain is None:
        gain = oracle.min_gain(mw, MW, W, **kw)
    return mw, MW, W, float(gain)


_logs = {}


def logs_of(name):
    """(case, per event: (scan log, breakpoints, counters)) -- cached, the CPU and GPU tests share it."""
    if name not in _logs:
        case = CASES[name]()
        mw, MW, W, gain = split_kw(case["kw"])
        _logs[name] = case, [oracle.scan_log(a, mw, MW, W, gain=gain) for a in case["arrays"]]
    return _logs[name]


# ------------------------------------------------------------------------------------------- the precondition
def variances(c, c2, s, e):
    """var_c(s, e) for arrays of (s, e) in the reference's operations (cparsers.pyx:31-38), no FMA."""
    s = np.asarray(s, np.int64)
    e = np.asarray(e, np.int64)
    n = (e - s).astype(np.float64)
    lo1 = np.where(s > 0, c[np.maximum(s - 1, 0)], 0.0)
    lo2 = np.where(s > 0, c2[np.maximum(s - 1, 0)], 0.0)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        m = (c[e - 1] - lo1) / n
        return (c2[e - 1] - lo2) / n - m * m


def operands(c, c2, ps, pe, i):
    """{(n1, V1), (n2, V2)} of candidate i as a sorted tuple of (n, bits of V)."""
    v1 = variances(c, c2, [ps], [i])[0]
    v2 = variances(c, c2, [i], [pe])[0]
    return tuple(sorted([(i - ps, np.float64(v1).view(np.int64).item()), (pe - i, np.float64(v2).view(np.int64).item())]))


def check_record(r, c, c2, mw, gain):
    """Why the decision of scan record r cannot depend on the rounding of `log`; raises AssertionError otherwise.
    Returns the kind: 'margin', 'inf', 'nan' or 'tie'."""
    g, ps, pe = r["gains"], r["ps"], r["pe"]
    ok = ~np.isnan(g)
    if not ok.any():
        assert r["x"] == -1
        return "nan"
    best = r["best"]
    if r["x"] < 0:
        assert best == -np.inf or gain - best >= REQUIRED, (ps, pe, best, gain)
        return "inf" if best == -np.inf else "margin"
    if best == np.inf:
        return "inf"
    assert best - gain >= REQUIRED, (ps, pe, best, gain)
    near = np.flatnonzero(ok & (g > best - REQUIRED))
    if len(near) == 1:
        return "margin"
    # every candidate that close must be an exact tie with identical operands
    want = operands(c, c2, ps, pe, r["best_i"])
    for j in near:
        i = ps + mw + int(j)
        assert g[j] == best and operands(c, c2, ps, pe, i) == want, (ps, pe, r["best_i"], i, best - g[j])
    return "tie"


def kinds_of(name):
    case, per_event = logs_of(name)
    mw, MW, W, gain = split_kw(case["kw"])
    out = []
    for a, (log, _, _) in zip(case["arrays"], per_event):
        c, c2 = oracle.cumsum(a)
        out.append([check_record(r, c, c2, mw, gain) for r in log])
    return out


def warp_of(ps, pe, mw, i):
    """Warp of k3_split whose piece holds candidate i of the only window of a level (chunks of 32 candidates,
    contiguous equal shares over the 4 warps)."""
    nch = (pe - ps - 2 * mw + 1 + 31) // 32
    per = (nch + 3) // 4
    return ((i - ps - mw) // 32) // per


def cta_of(ps, mw, i):
    """CTA of the k3_spine cluster that screens candidate i (4 CTAs x 512 threads, round-robin)."""
    return ((i - ps - mw) % 2048) // 512


def ties(name):
    case, per_event = logs_of(name)
    mw = split_kw(case["kw"])[0]
    out = []
    for e, (log, _, _) in enumerate(per_event):
        for r in log:
            g = r["gains"]
            if r["x"] >= 0 and np.isfinite(r["best"]):
                tied = np.flatnonzero(g == r["best"])
                if len(tied) > 1:
                    out.append((e, r, [r["ps"] + mw + int(j) for j in tied]))
    return out


def level_widths(log, n, mw, MW, W):
    """The local level-by-level search of k3_split replayed with the logged decisions: per level, the number of
    windows and the number of those whose interval's window loop had already advanced (ps > s)."""
    x_of = {(r["ps"], r["pe"]): r["x"] for r in log}

    def place(s, e, ps, out):          # k3_place: up to the next scannable window
        while True:
            if ps >= e - 2 * mw:
                if e - s > MW:
                    x = min(s + MW, e - mw)
                    for a, b in ((s, x), (x, e)):
                        if b - a > 2 * mw or b - a > MW:
                            place(a, b, a, out)
                return
            if ps > s + MW:
                s = ps = min(s + MW, e - mw)
                continue
            pe = min(ps + W, e)
            if pe - ps <= 2 * mw:
                ps = min(ps + W // 2, e)
                continue
            out.append((s, e, ps))
            return

    level, widths = [], []
    place(0, n, 0, level)
    while level:
        widths.append((len(level), sum(ps > s for s, _, ps in level)))
        nxt = []
        for s, e, ps in level:
            pe = min(ps + W, e)
            x = x_of[(ps, pe)]
            if x >= 0:
                for a, b in ((s, x), (x, e)):
                    if b - a > 2 * mw or b - a > MW:
                        place(a, b, a, nxt)
            else:
                place(s, e, min(ps + W // 2, e), nxt)
        level = nxt
    return widths


def _hi(x):
    """High 32-bit word of a double, signed (__double2hiint)."""
    return int(np.float64(x).view(np.int64)) >> 32


def _side_ok(S, Q, n, ebase):
    """k3_side's validity test restated exactly: r = fl(1/n), m = fl(S r), m2 = fl(m m), V = Q r - m2 rounded once
    (the fma), x = (exponent field of V) - ebase as unsigned <= 254, and the ratio test on the high words:
    hi(m2) - hi(V) < 24 << 20 in 32-bit signed arithmetic."""
    r = 1.0 / n
    m = S * r
    m2 = m * m
    if np.isfinite(Q) and np.isfinite(m2):
        V = float(Fraction(Q) * Fraction(r) - Fraction(m2))
    else:
        with np.errstate(invalid="ignore", over="ignore"):
            V = float(np.float64(Q) * np.float64(r) - np.float64(m2))
    vh = _hi(V)
    x = ((vh >> 20) - ebase) & 0xffffffff
    d = ((_hi(m2) - vh + 2 ** 31) % 2 ** 32) - 2 ** 31
    return x <= 254 and d < (24 << 20)


def screen_flags(c, c2, ps, pe, mw):
    """pp_debug_screen's `ok` per candidate ps+mw .. pe-mw, restated: the window's ebase (k3_window_ebase of its
    reference variance) and both sides' validity tests."""
    at = lambda p: (0.0, 0.0) if p < 0 else (float(c[p]), float(c2[p]))
    lo, hi = at(ps - 1), at(pe - 1)
    e = _hi(variances(c, c2, [ps], [pe])[0]) >> 20
    ebase = e - 127
    out = np.zeros(pe - 2 * mw - ps + 1, bool)
    if not 128 <= e <= 1919:
        return out
    for j, i in enumerate(range(ps + mw, pe - mw + 1)):
        mid = at(i - 1)
        out[j] = _side_ok(mid[0] - lo[0], mid[1] - lo[1], i - ps, ebase) and \
            _side_ok(hi[0] - mid[0], hi[1] - mid[1], pe - i, ebase)
    return out


def screen_windows(name, per_event_max=3):
    """(event, ps, pe, restated ok flags) of the first window scans of every event of a case."""
    case, per_event = logs_of(name)
    mw = split_kw(case["kw"])[0]
    out = []
    for e, (a, (log, _, _)) in enumerate(zip(case["arrays"], per_event)):
        c, c2 = oracle.cumsum(a)
        for r in log[:per_event_max]:
            out.append((e, r["ps"], r["pe"], screen_flags(c, c2, r["ps"], r["pe"], mw)))
    return out


def check_target(name):
    """Each case reaches what its name says."""
    case, per_event = logs_of(name)
    mw = split_kw(case["kw"])[0]
    logs = [log for log, _, _ in per_event]
    if name.startswith("mirror"):
        t = ties(name)
        assert t, "no exact tie is the window maximum"
        if name == "mirror_far":
            assert any(warp_of(r["ps"], r["pe"], mw, i[0]) != warp_of(r["ps"], r["pe"], mw, i[-1])
                       for _, r, i in t if r["ps"] == 0)
        if name == "mirror_spine":
            assert len(case["arrays"][0]) > 10240
            assert any(r["ps"] == 0 and cta_of(0, mw, i[0]) != cta_of(0, mw, i[-1]) for _, r, i in t)
    elif name == "inf_gains":
        assert max(r["n_posinf"] for log in logs for r in log) >= 2
        assert any(r["n_nan"] == len(r["gains"]) for log in logs for r in log)
        assert any(r["x"] >= 0 and r["best"] == np.inf and r["n_posinf"] >= 2 for log in logs for r in log)
    elif name in ("nonfinite", "extreme"):
        assert any(r["n_nan"] > 0 for log in logs for r in log)
        assert any(r["x"] >= 0 for log in logs for r in log)
    elif name == "crowded":
        assert max(r["n_near"] for log in logs for r in log) >= 256
        assert ties(name)
        # every candidate of the crowded windows passes the validity test: an exact full scan ([7]) of k3_split can
        # only come from the overflow of the exact-evaluation requests
        for e, ps, pe, ok in screen_windows(name):
            if len(ok) >= 256:
                assert ok.all(), (e, ps, pe)
    elif name == "full_levels":
        mw, MW, W, _ = split_kw(case["kw"])
        for a, log in zip(case["arrays"], logs):
            # a level past the 128-window list that holds an interval whose window loop has advanced
            assert any(n > 128 and adv > 0 for n, adv in level_widths(log, len(a), mw, MW, W))
    elif name == "validity":
        assert any(r["x"] >= 0 for log in logs for r in log)
        flags = {e: [] for e in range(len(case["arrays"]))}
        for e, ps, pe, ok in screen_windows(name):
            flags[e].append(ok)
        mixed = lambda e: any(ok.any() and not ok.all() for ok in flags[e])
        assert all(ok.all() for ok in flags[0])                       # (S/n)^2 / V ~ 2^22: every candidate valid
        assert mixed(1)                                               # ~ 2^24: both sides of the ratio test
        assert not any(ok.any() for ok in flags[2])                   # ~ 2^26: none
        assert mixed(3) and mixed(4)                                  # variances beyond ebase +- 127
        assert not any(ok.any() for ok in flags[5] + flags[6])        # the window's own variance is rejected


# ------------------------------------------------------------------------------------------------ CPU tests
def test_scan_log_equals_statsplit():
    """The scan log walks the same recursion as the C oracle: same breakpoints, candidates and scans."""
    from conftest import SCORING_CASES
    from pypore_b200 import synth
    events = [(synth.make_long_event(n, seed=s, tier=t).astype(np.float64), kw)
              for n, s, t, kw in SCORING_CASES.values()]
    x = synth.make_long_event(300000, seed=100, tier="A").astype(np.float64)
    events.append((x[:120000], dict(min_width=100, max_width=20000, window_width=10000)))
    for name in CASES:
        case = CASES[name]()
        events += [(a, case["kw"]) for a in case["arrays"][:2]]
    for a, kw in events:
        mw, MW, W, gain = split_kw(kw)
        _, bp, info = oracle.scan_log(a, mw, MW, W, gain=gain)
        want, winfo = oracle.statsplit(a, mw, MW, W, gain=gain, return_info=True)
        assert np.array_equal(bp, want)
        assert (info["ncand"], info["nscan"]) == (winfo["ncand"], winfo["nscan"])


@pytest.mark.parametrize("name", sorted(CASES))
def test_every_decision_is_robust(name):
    kinds = kinds_of(name)
    assert sum(len(k) for k in kinds) > 0
    check_target(name)
    flat = [k for ks in kinds for k in ks]
    if name.startswith("mirror") or name == "crowded":
        assert "tie" in flat
    if name in ("inf_gains",):
        assert "inf" in flat and "nan" in flat


def test_operand_identity_is_what_makes_a_tie_exact():
    """The restated operands see a difference of one ulp in a variance (the precondition is not vacuous)."""
    a = mirror(_levels(rng(1), (150, 250), (100.0, 80.0), 1.0))
    c, c2 = oracle.cumsum(a)
    n = len(a)
    assert operands(c, c2, 0, n, 150) == operands(c, c2, 0, n, n - 150)
    b = a.copy()
    b[-1] += 2.0 ** -5
    c, c2 = oracle.cumsum(b)
    assert operands(c, c2, 0, n, 150) != operands(c, c2, 0, n, n - 150)


# ------------------------------------------------------------------------------------------------ GPU tests
def put(ctx, kind, arrays):
    if kind == "flat64":
        ctx.upload_events_f64(arrays)
        return
    starts, pos = [], 0
    for i, a in enumerate(arrays):
        s = pos + 1 + (i % 8)
        starts.append(s)
        pos = s + len(a)
    dt = np.float32 if kind == "trace32" else np.float64
    buf = np.full(pos + 9, np.nan, dt)
    for s, a in zip(starts, arrays):
        buf[s:s + len(a)] = a
    if kind == "trace32":
        ctx.upload_trace(buf)
    else:
        ctx.upload_trace_f64(buf)
    ctx.set_events(np.asarray(starts, np.int64), np.asarray([len(a) for a in arrays], np.int64))


def kinds_for(arrays):
    with np.errstate(over="ignore"):
        f32 = all(np.array_equal(a.astype(np.float32).astype(np.float64), a, equal_nan=True) for a in arrays)
    return ["flat64", "trace64"] + (["trace32"] if f32 else [])


def modes(long_events):
    """(name, {option: value}) of the run matrix; option 0 screen, 1 spine, 2 CTAs, 3 kernel (1 = k3_flow)."""
    m = [("split", {}), ("split_exact", {0: 0}), ("flow", {3: 1}), ("flow_exact", {3: 1, 0: 0}),
         ("ctas1", {2: 1}), ("ctas3", {2: 3}), ("ctas148", {2: 148})]
    if long_events:
        m += [("nospine", {1: 0}), ("nospine_exact", {1: 0, 0: 0}), ("nospine_flow", {1: 0, 3: 1})]
    return m


def run_mode(ctx, opts, mw, MW, W, gain):
    """One split search with the options `opts`; the context's own values are restored afterwards.  Modes that do
    not name the kernel run k3_split."""
    opts = {3: 0, **opts}
    saved = {k: ctx.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        n = ctx.statsplit(mw, MW, W, gain)
        return ctx.segments(n, stats=False), ctx.split_counters()
    finally:
        for k, v in saved.items():
            ctx.set_option(k, v)


def expected_tables(per_event, arrays):
    ev, st, en = [], [], []
    for e, ((_, bp, _), a) in enumerate(zip(per_event, arrays)):
        edges = np.concatenate(([0], bp, [len(a)]))
        ev.append(np.full(len(edges) - 1, e))
        st.append(edges[:-1])
        en.append(edges[1:])
    return np.concatenate(ev), np.concatenate(st), np.concatenate(en)


def check_window_gains(ctx, case, per_event, mw):
    """pp_window_gains on every logged window against the C oracle's gains: NaN and +-inf at the same places,
    finite gains within 8u (|tot| + |low| + |high|)."""
    for e, (a, (log, _, _)) in enumerate(zip(case["arrays"], per_event)):
        if not log:
            continue
        c, c2 = oracle.cumsum(a)
        ps = np.array([r["ps"] for r in log], np.int32)
        pe = np.array([r["pe"] for r in log], np.int32)
        got = ctx.window_gains(e, ps, pe, mw)
        for r, g in zip(log, got):
            w = r["gains"]
            assert np.array_equal(np.isnan(g), np.isnan(w)), (e, r["ps"])
            inf = np.isinf(w)
            assert np.array_equal(g[inf], w[inf]) and not np.isinf(g[~inf]).any(), (e, r["ps"])
            f = np.isfinite(w)
            i = np.arange(r["ps"] + mw, r["pe"] - mw + 1)
            with np.errstate(divide="ignore", invalid="ignore"):
                tot = (r["pe"] - r["ps"]) * np.log(variances(c, c2, [r["ps"]], [r["pe"]])[0])
                low = (i - r["ps"]) * np.log(variances(c, c2, np.full(len(i), r["ps"]), i))
                high = (r["pe"] - i) * np.log(variances(c, c2, i, np.full(len(i), r["pe"])))
            bound = 8 * U * (abs(tot) + np.abs(low) + np.abs(high))
            assert np.all(np.abs(g[f] - w[f]) <= bound[f]), (e, r["ps"], np.max(np.abs(g[f] - w[f]) - bound[f]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_device_decisions(ctx, name):
    case, per_event = logs_of(name)
    mw, MW, W, gain = split_kw(case["kw"])
    arrays = case["arrays"]
    w_ev, w_st, w_en = expected_tables(per_event, arrays)
    ncand = sum(info["ncand"] for _, _, info in per_event)
    nscan = sum(info["nscan"] for _, _, info in per_event)
    long_events = max(len(a) for a in arrays) > 10240
    branches = {}
    for kind in kinds_for(arrays):
        put(ctx, kind, arrays)
        for mode, opts in modes(long_events):
            tab, cnt = run_mode(ctx, opts, mw, MW, W, gain)
            where = (name, kind, mode)
            assert np.array_equal(tab["event"], w_ev), where
            assert np.array_equal(tab["start"], w_st), where
            assert np.array_equal(tab["end"], w_en), where
            assert (cnt["candidates"], cnt["scans"]) == (ncand, nscan), (where, cnt, ncand, nscan)
            if 0 in opts:
                assert cnt["sure"] == cnt["multi"] == cnt["full"] == 0, (where, cnt)
            branches[(kind, mode)] = cnt
    put(ctx, "flat64", arrays)
    ctx.statsplit(mw, MW, W, gain)
    check_window_gains(ctx, case, per_event, mw)
    # the branches each family is built for
    b, f = branches[("flat64", "split")], branches[("flat64", "flow")]
    if name in ("mirror_short", "mirror_far"):
        assert b["multi"] > 0 and f["multi"] > 0, (b, f)
    if name == "mirror_spine":
        assert b["multi"] > 0 and branches[("flat64", "nospine")]["multi"] > 0, b
    if name in ("inf_gains", "nonfinite", "extreme"):
        assert b["full"] > 0 and f["full"] > 0, (b, f)
    if name == "crowded":
        # every candidate is valid (test_screen_validity_flags): k3_split's full scans come from the overflow of the
        # exact-evaluation requests; k3_flow has no request list and takes the argmax
        assert b["full"] > 0 and f["multi"] > 0, (b, f)
    if name == "full_levels":
        assert b["sure"] > 0 and b["full"] > 0, b
    if name == "validity":
        assert b["full"] > 0 and b["sure"] > 0 and f["full"] > 0, (b, f)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["validity", "crowded"])
def test_screen_validity_flags(ctx, name):
    """pp_debug_screen's validity flags equal the exact restatement of k3_side on the first windows of every event,
    and where a candidate is valid its screened value is within the bound of the reference's fl(low + high)."""
    case, _ = logs_of(name)
    mw, MW, W, gain = split_kw(case["kw"])
    ctx.upload_events_f64(case["arrays"])
    ctx.statsplit(mw, MW, W, gain)
    for e, ps, pe, want in screen_windows(name):
        hs, he, ok, eps = ctx.debug_screen(e, ps, pe, mw)
        assert np.array_equal(ok, want), (e, ps, pe, np.flatnonzero(ok != want)[:5])
        if ok.any():
            assert np.all(np.abs(hs[ok] - he[ok]) <= eps), (e, ps, pe, np.max(np.abs(hs[ok] - he[ok])), eps)


@pytest.mark.gpu
def test_min_gain_on_an_exact_tie(ctx):
    """min_gain equal to the tied gain: no split (strict '>'); one ulp below it: the lower tied index.  The gain is
    the device's own (pp_window_gains), so the comparison does not depend on the oracle's `log`."""
    mw = 100
    r = rng(8)
    arrays = []
    for a in (110, 125, 140):       # events of 3 mw: one window, both children leaves
        arrays.append(mirror(_levels(r, (a, 150 - a), (100.0, 80.0), 0.5)))
    for a in arrays:
        c, c2 = oracle.cumsum(a)
        n = len(a)
        g = oracle.scan_log(a, mw, 1000000, n, gain=-np.inf)[0][0]["gains"]
        j = int(np.argmax(g))
        i, k = mw + j, n - (mw + j)
        assert g[n - 2 * mw - j] == g[j] and operands(c, c2, 0, n, i) == operands(c, c2, 0, n, k)
        assert np.sort(g)[-3] < g[j] - REQUIRED
    ctx.upload_events_f64(arrays)
    ctx.statsplit(mw, 1000000, 300, 0.0)
    dev = [ctx.window_gains(e, [0], [len(a)], mw)[0] for e, a in enumerate(arrays)]
    for e, (a, g) in enumerate(zip(arrays, dev)):
        n = len(a)
        j = int(np.argmax(g))
        best = float(g[j])
        assert g[n - 2 * mw - j] == best
        for mg, want in ((best, []), (float(np.nextafter(best, -np.inf)), [min(mw + j, n - mw - j)])):
            for opts in ({}, {0: 0}, {3: 1}, {3: 1, 0: 0}):
                ctx.upload_events_f64([a])
                tab, _ = run_mode(ctx, opts, mw, 1000000, n, mg)
                assert list(tab["start"][1:]) == want, (e, mg, opts)
