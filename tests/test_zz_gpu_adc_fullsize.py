"""The BASELINE traces as int16 ADC counts at full size: c2 (bench.py's workload, 60 M samples) streamed through
pp_pipeline_host_adc16 with host tables, and c1, hash to the REAL reference's tables (tests/golden/c2_full.npz,
tests/golden/bench_configs.npz).  Tier A is k/32 with |k| < 2^15, so the counts k with scale 1/32 decode to exactly
the float32 trace's values."""
import numpy as np
import pytest

from conftest import load_golden, sha
from pypore_b200 import synth
from pypore_b200.adc import AdcTrace
from pypore_b200.parsers import statsplit_min_gain

pytestmark = pytest.mark.gpu

RULES = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)


def as_counts(ctx, x):
    k = np.round(x.astype(np.float64) * 32)
    assert np.abs(k).max() < 2 ** 15
    counts = ctx.pinned_empty(len(x), np.int16)
    counts[:] = k
    t = AdcTrace(counts, 1.0 / 32, 0.0)
    assert np.array_equal(t.decode(), x.astype(np.float64))
    return t


def hashes(r):
    es, el = r["event_table"]
    t = r["segment_table"]
    ev = np.stack([np.asarray(es, np.int64), np.asarray(el, np.int64)], axis=1)
    rows = np.stack([np.asarray(t["event"]).astype(np.int64), np.asarray(t["start"], np.int64),
                     np.asarray(t["end"], np.int64)], axis=1)
    return sha(ev), sha(rows)


def test_c2_counts_streamed_hash_to_the_reference(ctx):
    g = load_golden("c2_full.npz")
    x = synth.make_trace(5000, seed=1, tier="A")
    assert len(x) == int(g["samples"])
    t = as_counts(ctx, x)
    gain = statsplit_min_gain(**SPLIT)[3]
    r = ctx.pipeline(110.0, min_gain=gain, host_trace=t, export=True, **SPLIT, **RULES)
    assert r["events"] == int(g["events"]) and r["segments"] == int(g["default_segments"])
    assert hashes(r) == (str(g["events_sha"]), str(g["default_sha"]))


def test_c1_counts_hash_to_the_reference(ctx):
    g = load_golden("bench_configs.npz")
    x = synth.make_trace(500, seed=0, tier="A")
    assert len(x) == int(g["c1_samples"])
    t = as_counts(ctx, x)
    gain = statsplit_min_gain(**SPLIT)[3]
    r = ctx.pipeline(110.0, min_gain=gain, host_trace=t, export=True, **SPLIT, **RULES)
    assert (r["events"], r["segments"]) == (int(g["c1_events"]), int(g["c1_segments"]))
    assert ctx.split_counters()["candidates"] == int(g["c1_candidates"])
    assert hashes(r) == (str(g["c1_events_sha"]), str(g["c1_segments_sha"]))
