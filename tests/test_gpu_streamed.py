"""The streamed host pipeline (pp_pipeline_host, pp_pipeline_host_tables, pp_pipeline_host_adc16) against the resident
pipeline and the oracle, on traces that are longer than one chunk: long events spanning several chunks, crossings and
non-finite samples on chunk boundaries, every rule shape, every split option, both sample sources, the run-table
overflow redo and HMM merges after a streamed export.  The cases are built in tests/streamed_cases.py;
tests/test_streamed_cases_cpu.py checks that each one reaches what it was built for."""
import numpy as np
import pytest

import oracle
import streamed_cases as sc
from oracle import hmm as hmm_oracle
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import File
from pypore_b200.parsers import RuleSet, SpeedyStatSplit, lambda_event_parser

pytestmark = pytest.mark.gpu

COUNTS = ("runs", "events", "event_samples", "segments")


@pytest.fixture(scope="module")
def oracle_cache():
    return {}


def oracle_of(cache, case):
    if case.oracle_key not in cache:
        cache[case.oracle_key] = sc.oracle_tables(case)
    return cache[case.oracle_key]


@pytest.fixture
def options(ctx):
    """Set device options (id -> value) for one test; the values read before are restored afterwards."""
    saved = {}

    def apply(opts):
        for k, v in opts.items():
            saved.setdefault(k, ctx.get_option(k))
            ctx.set_option(k, v)
    yield apply
    for k, v in saved.items():
        ctx.set_option(k, v)


def bits_equal(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def same_nan_or_bits(a, b):
    """Equal bit for bit where finite or infinite, NaN at the same rows."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


def resident(ctx, case, **over):
    if isinstance(case.x, AdcTrace):
        ctx.upload_trace_adc16(case.x)
    else:
        ctx.upload_trace(case.x)
    r = ctx.pipeline(**dict(case.pipeline_kw(), **over))
    return tables(ctx, r)


def tables(ctx, r):
    ev = ctx.events(r["events"])
    return dict(counts={k: r[k] for k in COUNTS}, ev=ev, seg=ctx.segments(r["segments"]), ctr=ctx.split_counters())


def streamed(ctx, case, chunk, export, **over):
    r = ctx.pipeline(host_trace=case.x, chunk_samples=chunk, export=export, **dict(case.pipeline_kw(), **over))
    t = tables(ctx, r)
    if export:    # the exported host rows are the device tables
        es, el = r["event_table"]
        assert np.array_equal(es, t["ev"][0]) and np.array_equal(el, t["ev"][1])
        assert set(r["segment_table"]) == set(t["seg"])
        for k, v in r["segment_table"].items():
            assert np.array_equal(v, t["seg"][k], equal_nan=True), k
    return t


def assert_same(got, want, where):
    assert got["counts"] == want["counts"], where
    assert np.array_equal(got["ev"][0], want["ev"][0]) and np.array_equal(got["ev"][1], want["ev"][1]), where
    assert set(got["seg"]) == set(want["seg"])
    for k in got["seg"]:
        assert np.array_equal(got["seg"][k], want["seg"][k], equal_nan=True), (where, k)
    # The work the split search does is fixed by the recursion.  How a screened window is decided (exact, sure, multi,
    # full) and the task count are not: k3_split / k3_flow hand intervals to idle CTAs ("few" mode) when a launch starts
    # with fewer than two tasks per CTA, which each chunk's launch may, and how many CTAs wait at that moment is a
    # matter of timing.  That changes which windows share a level, hence the request-list overflows (full) and the
    # multi-contender resolutions.
    for k in ("candidates", "scans", "seq_redo"):
        assert got["ctr"][k] == want["ctr"][k], (where, k, got["ctr"], want["ctr"])


def assert_oracle(got, want, where):
    assert np.array_equal(got["ev"][0], want["ev_start"]) and np.array_equal(got["ev"][1], want["ev_len"]), where
    for k in ("event", "start", "end"):
        assert np.array_equal(np.asarray(got["seg"][k], np.int64), want[k]), (where, k)
    for k in ("min", "max"):
        assert same_nan_or_bits(got["seg"][k], want[k]), (where, k)
    for k in ("mean", "std"):
        assert np.allclose(got["seg"][k], want[k], rtol=1e-9, atol=0, equal_nan=True), (where, k)


def check_case(ctx, cache, case, oracle_check=True):
    want = resident(ctx, case)
    if oracle_check:
        assert_oracle(want, oracle_of(cache, case), (case.name, "resident"))
    for chunk in case.chunks:
        runs = [streamed(ctx, case, chunk, export) for export in (False, True)]
        for export, got in zip((False, True), runs):
            where = (case.name, chunk, export)
            assert_same(got, want, where)
            if oracle_check:
                assert_oracle(got, oracle_of(cache, case), where)
    return want


LONG = [n for n in sc.cases() if n.startswith("long_")]
OPTION = [n for n in sc.cases() if n.startswith("option_")]
PREFIX = [n for n in sc.cases() if n.startswith("prefix_")]
EDGES = [n for n in sc.cases() if n.startswith(("edges_", "dense"))]
RULES = [n for n in sc.cases() if n.startswith("rules_")]


@pytest.mark.parametrize("name", LONG)
def test_long_events_every_chunking(ctx, oracle_cache, name):
    """Every length class of the split stages, events longer than three chunks, the open long last run; every chunk
    size from 1 (rounded to 4096) to n (resident fallback); tier B redoes its prefix sums in every chunk."""
    case = sc.cases()[name]
    want = check_case(ctx, oracle_cache, case)
    if name == "long_B":
        assert want["ctr"]["seq_redo"] > 0


@pytest.mark.parametrize("name", OPTION)
def test_split_options(ctx, oracle_cache, options, name):
    case = sc.cases()[name]
    options(case.options)
    check_case(ctx, oracle_cache, case)


@pytest.mark.parametrize("name", PREFIX)
def test_prefix_modes(ctx, oracle_cache, name):
    """SEQUENTIAL always equals the oracle; PARALLEL does where the data pass the exactness proof (tier A) and
    otherwise equals the resident PARALLEL run."""
    case = sc.cases()[name]
    check_case(ctx, oracle_cache, case, oracle_check=not name.startswith("prefix_parallel_B"))


@pytest.mark.parametrize("name", sorted(sc.ADC_SOURCES))
def test_adc_sources(ctx, oracle_cache, name):
    check_case(ctx, oracle_cache, sc.cases()[name])


@pytest.mark.parametrize("name", EDGES)
def test_chunk_edges(ctx, oracle_cache, name):
    check_case(ctx, oracle_cache, sc.cases()[name])


@pytest.mark.parametrize("name", RULES)
def test_rule_shapes(ctx, oracle_cache, name):
    check_case(ctx, oracle_cache, sc.cases()[name])


def test_run_table_overflow_redo(ctx, oracle_cache):
    """More runs than the streamed call reserves: pp_pipeline_host redoes the whole trace resident, the exporting call
    falls back to the device tables; both equal the resident run and the oracle."""
    case = sc.Case("overflow", sc.overflow_trace(), rules=sc.DENSE_RULES, split="dense", chunks=(1 << 18,))
    want = check_case(ctx, oracle_cache, case)
    assert want["counts"]["runs"] > case.n // 256 + 4096


def test_filtered_call_runs_resident(ctx):
    """With a filter the streamed call runs resident by design: the same tables for a small chunk size."""
    from pypore_b200.DataTypes import bessel_coefficients
    case = sc.cases()["long_A"]
    filt = bessel_coefficients(1, 2000.0, 1e5)
    want = resident(ctx, case, filter_ba=filt)
    got = streamed(ctx, case, 65536, False, filter_ba=filt)
    assert_same(got, want, "filtered")


def test_hmm_merge_after_streamed_export(ctx):
    """Decoding and merging the tables a chunked export left on the device gives what it gives after the resident
    pipeline, and the merge equals the oracle's on the device's states."""
    case = sc.cases()["long_A_psps10"]
    model = sc.hmm_model()
    out = []
    for run in ("resident", "streamed"):
        t = resident(ctx, case) if run == "resident" else streamed(ctx, case, 65536, True)
        n_ev, n_seg = t["counts"]["events"], t["counts"]["segments"]
        assert ctx.hmm_decode(model, "forward") == n_seg
        lp_f, _ = ctx.hmm_download(n_ev)
        assert ctx.hmm_decode(model, "viterbi") == n_seg
        lp_v, st = ctx.hmm_download(n_ev, n_seg)
        n_m = ctx.hmm_decode(model, "viterbi", merge=True)
        lp_m, st_m = ctx.hmm_download(n_ev, n_m)
        out.append(dict(t=t, lp_f=lp_f, lp_v=lp_v, st=st, lp_m=lp_m, st_m=st_m, seg_m=ctx.segments(n_m)))
    a, b = out
    assert bits_equal(a["lp_f"], b["lp_f"]) and bits_equal(a["lp_v"], b["lp_v"]) and bits_equal(a["lp_m"], b["lp_m"])
    assert np.array_equal(a["st"], b["st"]) and np.array_equal(a["st_m"], b["st_m"])
    for k in a["seg_m"]:
        assert np.array_equal(a["seg_m"][k], b["seg_m"][k], equal_nan=True), k
    seg = b["t"]["seg"]
    e, s, t, q = hmm_oracle.hmm_merge(seg["event"], seg["start"], seg["end"], b["st"])
    assert len(e) < len(seg["event"])
    for name, want in (("event", e), ("start", s), ("end", t)):
        assert np.array_equal(b["seg_m"][name], want), name
    assert np.array_equal(b["st_m"], q)
    x = case.current()
    ws = b["t"]["ev"][0]
    base = ws[b["seg_m"]["event"]]
    m, sd, mn, mx = oracle.segment_stats(x, base + b["seg_m"]["start"], base + b["seg_m"]["end"])
    assert bits_equal(b["seg_m"]["min"], mn) and bits_equal(b["seg_m"]["max"], mx)
    assert np.allclose(b["seg_m"]["mean"], m, rtol=1e-9, atol=0) and np.allclose(b["seg_m"]["std"], sd, rtol=1e-9, atol=0)


# ---------------------------------------------------------------------------------------------------------------
# the public path: File.parse streams a trace longer than the default chunk
# ---------------------------------------------------------------------------------------------------------------
PSPS10 = dict(min_width=100, window_width=10000, prior_segments_per_second=10)


@pytest.fixture(scope="module")
def big():
    x = sc.big_trace()
    return x, sc.oracle_tables(sc.Case("big", x, split="psps10"))


def parse(trace, hmm=None):
    f = File(current=trace, timestep=1000. / 1e5)
    f.parse(parser=lambda_event_parser(threshold=110, rules=RuleSet(duration_gt=1000, min_gt=-0.5, max_lt=110)),
            segmenter=SpeedyStatSplit(**PSPS10), hmm=hmm)
    return f


def check_file(f, x64, want):
    et, st = f.event_table, f.segment_table
    assert np.array_equal(et["start"], want["ev_start"]) and np.array_equal(et["length"], want["ev_len"])
    for k in ("event", "start", "end"):
        assert np.array_equal(np.asarray(st[k], np.int64), want[k]), k
    for k in ("min", "max"):
        assert bits_equal(st[k], want[k]), k
    for k in ("mean", "std"):
        assert np.allclose(st[k], want[k], rtol=1e-9, atol=0), k
    ev = [x64[s:s + n] for s, n in zip(want["ev_start"], want["ev_len"])]
    assert bits_equal(et["min"], [v.min() for v in ev]) and bits_equal(et["max"], [v.max() for v in ev])
    assert np.allclose(et["mean"], [np.mean(v) for v in ev], rtol=1e-9, atol=0)
    assert np.allclose(et["std"], [np.std(v) for v in ev], rtol=1e-9, atol=0)


@pytest.mark.parametrize("source", ["float32", "adc"])
def test_file_parse_streams_a_trace_longer_than_the_default_chunk(big, source):
    x, want = big
    assert sc.streams(len(x), 0)
    trace = x if source == "float32" else sc.adc_of(x, 1.0 / 32)
    check_file(parse(trace), x.astype(np.float64), want)


def test_file_parse_hmm_merge_on_a_streamed_trace(big):
    x, want = big
    model = sc.hmm_model()
    plain, merged = parse(x), parse(x, hmm=model)
    pt, mt = plain.segment_table, merged.segment_table
    n_ev = len(plain.event_table["start"])
    b = np.searchsorted(pt["event"], np.arange(n_ev + 1))
    got = model.viterbi_many([pt["mean"][b[i]:b[i + 1]] for i in range(n_ev)])
    assert bits_equal(merged.event_table["log_probability"], [lp for lp, _ in got])
    e, s, t, q = hmm_oracle.hmm_merge(pt["event"], pt["start"], pt["end"], np.concatenate([st for _, st in got]))
    assert len(e) < len(pt["event"])
    for name, w in (("event", e), ("start", s), ("end", t), ("state", q)):
        assert np.array_equal(mt[name], w), name
    x64 = x.astype(np.float64)
    base = plain.event_table["start"][mt["event"]]
    m, sd, mn, mx = oracle.segment_stats(x64, base + mt["start"], base + mt["end"])
    assert bits_equal(mt["min"], mn) and bits_equal(mt["max"], mx)
    assert np.allclose(mt["mean"], m, rtol=1e-9, atol=0) and np.allclose(mt["std"], sd, rtol=1e-9, atol=0)
