"""The cases of tests/test_gpu_rows.py reach what they were built for (no GPU): the oracle finds exactly the designed
events and breakpoints, each row-locality case puts the same rows into tables whose mean row length lies on both sides
of K4_WIDE (so that a per-launch group width would differ), the rows' sums are order-sensitive, and the compaction
tables set bits on word and block edges."""
import numpy as np
import pytest

import oracle
import row_cases as rc
from oracle import hmm as hmm_oracle

SENSITIVE = 0.2     # the least fraction of order-sensitive rows in each case


def oracle_table(x64, ev_start, ev_len, split=rc.SPLIT, gain=rc.GAIN):
    e, s, t, _ = oracle.statsplit_events(x64, ev_start, ev_len, split["min_width"], split["max_width"],
                                         split["window_width"], gain=gain, threads=8)
    return e, s, t


def assert_table(got, want):
    for g, w, name in zip(got, want, ("event", "start", "end")):
        assert np.array_equal(g, w), name


def fraction_sensitive(rows):
    return np.mean([rc.order_sensitive(r) for r in rows])


@pytest.mark.parametrize("kind", rc.STREAM_KINDS)
@pytest.mark.parametrize("name", sorted(rc.STREAM_CASES))
def test_stream_traces_split_as_designed_and_cross_the_width(name, kind):
    make, chunks = rc.STREAM_CASES[name]
    tr = make(kind)
    runs = oracle.threshold_runs(tr.x64, rc.RULES["threshold"])
    keep = oracle.select_runs(tr.x64, runs, [lambda e: e.duration > rc.RULES["duration_gt"], lambda e: e.max < 110.0])
    assert np.array_equal(runs[0][keep], tr.ev_start) and np.array_equal(runs[1][keep], tr.ev_len)
    e, s, t = tr.table()
    assert_table(oracle_table(tr.x64, tr.ev_start, tr.ev_len), (e, s, t))
    assert rc.width(int(tr.ev_len.sum()), len(e)) == 8 and tr.ev_len.sum() / len(e) <= 256
    for chunk in chunks:
        assert rc.rounded(chunk) < tr.n                               # streamed, not run resident
        per, whole = rc.chunk_widths(tr, chunk)
        assert any(w is not None and w != whole for w in per), (chunk, per)
        if name == "long_then_short":
            assert per[0] == 32                                       # the first chunk holds long segments only
        else:                                                         # only an inner chunk crosses
            assert per[0] == whole and per[-1] == whole and 32 in per[1:-1], (chunk, per)
    rows = [tr.x64[a + b:a + c] for a, b, c in zip(tr.ev_start[e], s, t)]
    assert fraction_sensitive(rows) >= SENSITIVE
    if name == "long_then_short":
        first = rc.completed_by(tr, chunks[0])[0]
        assert len(first) and (tr.ev_len[first] / (np.array([len(b) for b in tr.bps])[first] + 1)).min() >= 2000
        assert first.max() < len(tr.ev_start) - 1


@pytest.mark.parametrize("kind", rc.SUBSET_KINDS)
def test_subsets_split_as_designed_and_cross_the_width(kind):
    p = rc.subset_events(kind)
    seg_w, ev_w = {}, {}
    for name, which in rc.subsets().items():
        e, s, t = p.table(which)
        assert_table(oracle_table(p.x64, p.start[which], p.length[which]), (e, s, t))
        total = int(p.length[which].sum())
        seg_w[name], ev_w[name] = rc.width(total, len(e)), rc.width(total, len(which))
    assert seg_w == ev_w == {"all": 8, "long": 32, "long_plus_one_short": 32}
    one = rc.subsets()["long_plus_one_short"][-1]
    assert p.length[one] < rc.K4_WIDE
    e, s, t = p.table(rc.subsets()["all"])
    assert fraction_sensitive([p.rows[a][b:c] for a, b, c in zip(e, s, t)]) >= SENSITIVE
    assert fraction_sensitive(p.rows) >= SENSITIVE
    if kind == "float64":   # not float32-representable
        assert not np.array_equal(p.rows[0].astype(np.float32).astype(np.float64), p.rows[0])


@pytest.mark.parametrize("kind", rc.SUBSET_KINDS)
def test_merge_events_merge_pairwise_across_the_width(kind):
    p = rc.merge_events(kind)
    which = np.arange(len(p.rows))
    e, s, t = p.table(which)
    assert_table(oracle_table(p.x64, p.start, p.length), (e, s, t))
    model = rc.merge_model()
    states = []
    for i in which:
        sel = e == i
        means = np.array([p.rows[i][a:b].mean() for a, b in zip(s[sel], t[sel])])
        _, st = hmm_oracle.hmm_viterbi(means, **model.params())
        states.append(np.asarray(st))
        assert list(st) == [q for q, k in rc.MERGE_PATTERN for _ in range(k)], i
    me, ms, mt, _ = hmm_oracle.hmm_merge(e, s, t, np.concatenate(states))
    assert_table((me, ms, mt), rc.merged_table(p))
    total = int(p.length.sum())
    assert rc.width(total, len(e)) == 8 and rc.width(total, len(me)) == 32
    kept = set(zip(me.tolist(), ms.tolist(), mt.tolist())) & set(zip(e.tolist(), s.tolist(), t.tolist()))
    assert len(kept) == len(p.rows)                                   # the singles are left as they were
    assert fraction_sensitive([p.rows[a][b:c] for a, b, c in zip(e, s, t)]) >= SENSITIVE


def test_compaction_edges_put_bits_on_word_and_block_edges():
    events, cuts = rc.compaction_edges()
    e, s, t, flat = rc.oracle_flat(events, rc.EDGE_SPLIT, rc.EDGE_GAIN)
    assert np.array_equal(flat, cuts)
    off = rc.flat_offsets(events)
    starts = set(off[:-1].tolist())
    inner = set(cuts.tolist()) - starts
    B = rc.CP_BLOCK_SAMPLES
    for group in (starts, inner):
        assert {f % 32 for f in group} >= {0, 31}                     # bit 0 and bit 31 of a word
    assert {B - 1} <= inner and {2 * B} <= inner                      # breakpoints at a block's last / first sample
    assert {3 * B - 1, 3 * B} <= starts                               # ... and event starts
    assert {1, 2, 3} <= set(np.diff(off).tolist())                    # events of 1, 2 and 3 samples

    alt = rc.alternating_events()
    _, _, _, flat = rc.oracle_flat(alt, rc.ALT_SPLIT, rc.ALT_GAIN)
    bits = np.zeros(int(rc.flat_offsets(alt)[-1]), bool)
    bits[flat] = True
    assert bits[:len(bits) // 32 * 32].reshape(-1, 32).all(axis=1).sum() >= 20   # words with all 32 bits set

    big, cuts = rc.big_flat_events()
    _, _, _, flat = rc.oracle_flat(big, rc.BIG_SPLIT, rc.BIG_GAIN)
    assert np.array_equal(flat, cuts)
    n = int(rc.flat_offsets(big)[-1])
    E = rc.CP_SCAN_BLOCKS * B
    assert n > 33554432 and -(-n // B) > rc.CP_SCAN_BLOCKS
    assert {E - 1, E + 100, E + 287} <= set(cuts.tolist()) and (cuts > E).sum() > 100
