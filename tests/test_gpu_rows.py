"""Row locality of compaction and segment statistics (K3c + K4): a row's statistics depend only on its own samples and
on where they sit in the trace or the flat event space, never on the other rows, the row range of a launch or the
length of the table.  Every column is compared bit for bit (NaN at the same rows) between runs that put the same rows
into different tables -- the resident pipeline and the streamed export at several chunk sizes, subsets of the placed
events, the tables before and after an HMM merge -- and every row also against the exact references of
tests/test_gpu_numerics.py and the oracle's event / start / end.  Then K4's own boundaries at every 16-byte phase on
every sample source, and the compaction tables on word, block and scan edges.  The cases are built in
tests/row_cases.py; tests/test_row_cases_cpu.py checks that each one reaches what it was built for (in particular that
the designed tables are the oracle's)."""
import numpy as np
import pytest

import row_cases as rc
from pypore_b200.adc import AdcTrace
from test_gpu_numerics import Content, check_stats, put, reference_stats, same_bits
from test_gpu_streamed import options  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

COLS = ("mean", "std", "min", "max")


def assert_rows_same(got, want, ig, iw, where):
    """Columns of rows ig of `got` bit for bit those of rows iw of `want`."""
    for k in COLS:
        a, b = np.asarray(got[k])[ig], np.asarray(want[k])[iw]
        if not same_bits(a, b):
            bad = np.flatnonzero((a != b) & ~(np.isnan(a) & np.isnan(b)))
            raise AssertionError("%s %s: %d of %d rows differ, first %s: %r != %r" %
                                 (where, k, len(bad), len(a), np.asarray(ig)[bad[:3]], a[bad[:3]], b[bad[:3]]))


def assert_exact(tab, rows, where):
    """Every row's statistics against the exact references (mean / std 1e-9, min / max bitwise)."""
    c = Content(rows=rows)
    check_stats(tab, reference_stats(c), c.lengths(), (where, "", ""), {})


def assert_table(tab, e, s, t, where):
    for name, want in (("event", e), ("start", s), ("end", t)):
        assert np.array_equal(np.asarray(tab[name], np.int64), want), (where, name)


# ------------------------------------------------------------------------------- streamed export against resident
def pipeline_kw():
    return dict(rc.RULES, min_gain=rc.GAIN, **rc.SPLIT)


def resident(ctx, tr):
    if isinstance(tr.x, AdcTrace):
        ctx.upload_trace_adc16(tr.x)
    else:
        ctx.upload_trace(tr.x)
    r = ctx.pipeline(**pipeline_kw())
    return r, ctx.events(r["events"]), ctx.segments(r["segments"])


@pytest.mark.parametrize("kind", rc.STREAM_KINDS)
@pytest.mark.parametrize("name", sorted(rc.STREAM_CASES))
def test_streamed_export_rows_equal_the_resident_run(ctx, name, kind):
    """Long segments first (or in an inner chunk only), short ones after: each chunk's K4 launch covers other rows
    than the resident launch over the whole table, yet every row has the same bits."""
    make, chunks = rc.STREAM_CASES[name]
    tr = make(kind)
    r, ev, want = resident(ctx, tr)
    e, s, t = tr.table()
    assert np.array_equal(ev[0], tr.ev_start) and np.array_equal(ev[1], tr.ev_len)
    assert_table(want, e, s, t, (name, kind, "resident"))
    base = tr.ev_start[e]
    assert_exact(want, [tr.x64[b + a:b + c] for b, a, c in zip(base, s, t)], (name, kind))
    every = np.arange(len(e))
    for chunk in chunks:
        got = ctx.pipeline(host_trace=tr.x, chunk_samples=chunk, export=True, **pipeline_kw())
        assert got["segments"] == r["segments"] and got["events"] == r["events"]
        tab = got["segment_table"]
        assert_table(tab, e, s, t, (name, kind, chunk))
        assert_rows_same(tab, want, every, every, (name, kind, chunk))


# ------------------------------------------------------------------------------- subsets of placed events
def split_and_stats(ctx):
    n = ctx.statsplit(rc.SPLIT["min_width"], rc.SPLIT["max_width"], rc.SPLIT["window_width"], rc.GAIN)
    ctx.segment_stats()
    return ctx.segments(n)


@pytest.mark.parametrize("kind", rc.SUBSET_KINDS)
def test_subset_rows_equal_the_rows_among_all_events(ctx, kind):
    """The same events at the same trace positions, with fewer or other neighbours: segment and event statistics of
    each event bit for bit what they are among all events."""
    p = rc.subset_events(kind)
    runs = {}
    for name, which in rc.subsets().items():
        p.upload(ctx, which)
        tab = split_and_stats(ctx)
        e, s, t = p.table(which)
        assert_table(tab, e, s, t, (kind, name))
        assert_exact(tab, [p.rows[which[i]][a:b] for i, a, b in zip(e, s, t)], (kind, name))
        evs = ctx.event_stats(len(which))
        assert_exact(evs, [p.rows[i] for i in which], (kind, name, "events"))
        runs[name] = (which, tab, evs, np.searchsorted(e, np.arange(len(which) + 1)))
    _, tab_all, evs_all, off_all = runs["all"]
    for name, (which, tab, evs, off) in runs.items():
        ig = np.arange(off[-1])
        iw = np.concatenate([np.arange(off_all[j], off_all[j + 1]) for j in which])
        assert_rows_same(tab, tab_all, ig, iw, (kind, name, "segments"))
        assert_rows_same(evs, evs_all, np.arange(len(which)), which, (kind, name, "events"))


# ------------------------------------------------------------------------------- HMM merge
@pytest.mark.parametrize("kind", rc.SUBSET_KINDS)
def test_merge_leaves_the_rows_it_does_not_touch(ctx, kind):
    """Pairs of near levels merge into rows of > 512 samples; the single segments between them keep their bits."""
    p = rc.merge_events(kind)
    which = np.arange(len(p.rows))
    p.upload(ctx, which)
    pre = split_and_stats(ctx)
    e, s, t = p.table(which)
    assert_table(pre, e, s, t, (kind, "pre"))
    n = ctx.hmm_decode(rc.merge_model(), "viterbi", merge=True)
    post = ctx.segments(n)
    me, ms, mt = rc.merged_table(p)
    assert_table(post, me, ms, mt, (kind, "post"))
    assert_exact(post, [p.rows[i][a:b] for i, a, b in zip(me, ms, mt)], (kind, "post"))
    key = {(a, b, c): i for i, (a, b, c) in enumerate(zip(e.tolist(), s.tolist(), t.tolist()))}
    ig = [i for i, k in enumerate(zip(me.tolist(), ms.tolist(), mt.tolist())) if k in key]
    iw = [key[(me[i], ms[i], mt[i])] for i in ig]
    assert len(ig) == len(p.rows)
    assert_rows_same(post, pre, np.array(ig), np.array(iw), (kind, "untouched"))


# ------------------------------------------------------------------------------- K4's own boundaries
def boundary_rows(rng):
    """float64 rows: the width boundary, one pass / two passes, both sides of the m1^2 > 1024 var redo."""
    rows = [0.3 + rng.normal(0.0, 1.0, n) for n in (511, 512, 513, 65536, 65537)]
    for n in (2000, 5000):                       # first sample 0, the rest near mu: m1^2 / var = 1024 (1 -+ 10 %)
        for f in (0.9, 1.1):
            r = 1024.0 * f
            mu = np.sqrt(r * (n - 1) / n / ((n - 1) ** 2 / n ** 2 - r * (n - 1) / n ** 2))
            rows.append(np.r_[0.0, mu + rng.normal(0.0, 1.0, n - 1)])
    return rows


def redo_ratio(row):
    d = row - row[0]
    m1 = d.mean()
    return m1 * m1 / (np.mean(d * d) - m1 * m1)


def special_rows(rng):
    """float32-exact rows: non-finite first samples (the shift falls back to 0), +-0.0 as the only extreme."""
    out = []
    for n in (300, 700):
        body = rng.normal(0.3, 1.0, n - 1).astype(np.float32).astype(np.float64)
        out += [np.r_[v, body] for v in (np.inf, -np.inf, np.nan)]
        pos = (np.abs(body) + 1.0).astype(np.float32).astype(np.float64)
        out.append(np.r_[-0.0, pos])                     # min is -0.0
        out.append(np.r_[-pos, 0.0])                     # max is +0.0
    return out


def boundary_contents():
    rng = np.random.RandomState(51)
    rows = boundary_rows(rng)
    for r in rows[5:]:
        f = redo_ratio(r) / 1024.0
        assert 0.85 < f < 0.95 or 1.05 < f < 1.15, f
    f32 = [r.astype(np.float32).astype(np.float64) for r in rows] + special_rows(rng)
    counts = [np.round((r - rc.ADC_OFFSET) / rc.ADC_SCALE) for r in rows]
    return {"float32": Content(rows=f32), "float64": Content(rows=rows),
            "adc": Content(counts=counts, scale=rc.ADC_SCALE, offset=rc.ADC_OFFSET)}


@pytest.mark.parametrize("family", ["float32", "float64", "adc"])
def test_k4_boundaries_every_phase_and_source(ctx, family):
    """Rows of 511 / 512 / 513 and 65,536 / 65,537 samples, on both sides of the two-pass redo, with a non-finite first
    sample and with +-0.0 extremes, at all eight 16-byte phases; NaN (ADC: int16 extremes) fills the elements in front
    of and behind every row and must not leak into it."""
    content = boundary_contents()[family]
    ref = reference_stats(content)
    lens = content.lengths()
    for kind in content.kinds():
        for phase in range(8 if kind != "flat64" else 1):
            put(ctx, kind, content, phase=phase)
            check_stats(ctx.event_stats(len(lens)), ref, lens, (family, kind, phase), {})


# ------------------------------------------------------------------------------- compaction edges
FLAT_TABLES = {"edges": (rc.compaction_edges, rc.EDGE_SPLIT, rc.EDGE_GAIN),
               "alternating": (rc.alternating_events, rc.ALT_SPLIT, rc.ALT_GAIN),
               "big": (rc.big_flat_events, rc.BIG_SPLIT, rc.BIG_GAIN)}


@pytest.fixture(scope="module")
def flat_tables():
    """name -> (events, split, gain, the oracle's event / start / end / flat start), each oracle run once."""
    out = {}
    for name, (make, split, gain) in FLAT_TABLES.items():
        events = make()
        events = list(events[0] if isinstance(events, tuple) else events)
        out[name] = (events, split, gain, rc.oracle_flat(events, split, gain))
    return out


def check_flat(ctx, kind, events, split, gain, want, where, idx=None):
    """The device's table of `events` placed as `kind` (packed float64 events, or a float64 trace with set_events:
    the flat event space is the same) equals the oracle's; the statistics of rows `idx` (all by default) equal the
    exact references."""
    put(ctx, kind, Content(rows=events))
    n = ctx.statsplit(split["min_width"], split["max_width"], split["window_width"], gain)
    ctx.segment_stats()
    tab = ctx.segments(n)
    e, s, t, _ = want
    assert n == len(e), where
    assert_table(tab, e, s, t, where)
    idx = np.arange(n) if idx is None else idx
    sub = {k: tab[k][idx] for k in COLS}
    assert_exact(sub, [events[e[i]][s[i]:t[i]] for i in idx], where)


@pytest.mark.parametrize("kind", ["flat64", "trace64"])
@pytest.mark.parametrize("screen", [1, 0])
def test_compaction_edges(ctx, options, flat_tables, screen, kind):
    """Bits 0 and 31 of a word, both sides of a 1,024-word block edge, events of 1-3 samples, words with all 32 bits
    set, and a table of more than 1,024 blocks (k3c_scan's carry); packed float64 events and the same events on a
    float64 trace; with the split screen on and off (the exact fallback)."""
    options({0: screen})
    for name, (events, split, gain, want) in flat_tables.items():
        idx = None
        if name == "big":       # every 17th row and the rows around the 1,024-block edge
            E = rc.CP_SCAN_BLOCKS * rc.CP_BLOCK_SAMPLES
            n = len(want[0])
            k = int(np.searchsorted(want[3], E))
            assert rc.flat_offsets(events)[-1] > E
            idx = np.unique(np.r_[np.arange(0, n, 17), np.arange(max(k - 3, 0), min(k + 3, n)), n - 1])
        check_flat(ctx, kind, events, split, gain, want, (name, kind, screen), idx)
