"""The cases of tests/test_gpu_streamed.py reach what they were built for (no GPU): length classes, crossings and
non-finite samples on rounded chunk boundaries, chunks that complete no event or more than 1,024 runs, the open long
last run, the rule shapes and the run-table overflow.  Everything is read off the oracle's run table and the chunk
grid pipeline_host_impl uses."""
import numpy as np
import pytest

import streamed_cases as sc


def selected(case):
    runs, keep = sc.oracle_runs(case)
    return runs, runs[0][keep], runs[1][keep]


def test_chunk_rounding_and_grid():
    assert [sc.rounded(c) for c in (1, 4095, 4096, 4096 * 37 + 1, 0)] == [4096, 4096, 4096, 4096 * 38, 16 << 20]
    s = np.array([0, 10, 4095, 4096, 8190])
    l = np.array([10, 4085, 1, 4094, 2])
    # runs ending at 10, 4095 (sample 4095 is in chunk 0), 4096 (in chunk 1), 8190, 8192 == n (the last chunk)
    assert list(sc.completions(8192, 4096, s, l)) == [0, 0, 1, 1, 1]
    assert sc.streams(8193, 8192) and not sc.streams(8192, 8192) and sc.chunk_count(8193, 4096) == 3


@pytest.mark.parametrize("tier", ["A", "B"])
def test_long_event_trace_reaches_every_length_class(tier):
    case = sc.cases()["long_" + tier]
    n = case.n
    runs, ws, wl = selected(case)
    assert len(ws) == len(sc.LONG_LAYOUT) + 1 and np.array_equal(wl, sc.LONG_LAYOUT + (sc.OPEN_LAST,))
    spine = (wl > sc.K3_CAP) & (wl <= sc.K2F_MAX_LEN)
    tiled = wl > sc.K2F_MAX_LEN
    assert spine.sum() >= 3 and tiled.sum() >= 6
    rem = wl[tiled] % sc.K2_TILE
    assert (rem == 0).any() and (rem == 1).any() and ((rem > 1)).any()   # last K2 tile full, one sample, ragged
    assert ws[-1] + wl[-1] == n and wl[-1] > sc.K2F_MAX_LEN             # a long open last run
    assert wl.max() <= 1500000
    for chunk in sc.TARGET_CHUNKS:
        C, K = sc.rounded(chunk), sc.chunk_count(n, chunk)
        assert sc.streams(n, chunk)
        done = sc.completions(n, chunk, ws, wl)
        per = np.bincount(done, minlength=K)
        assert wl.max() > 3 * C
        first = int(np.flatnonzero(per)[0])
        assert any(per[k] == 0 for k in range(first + 1, K - 1))    # intermediate chunks complete no event
        assert done[-1] == K - 1 and per[K - 1] == 1                # the open last run: only the final call
        # a spine event completed after a chunk that already completed events (ev_begin > 0), and a tiled event
        # completed after a chunk that already completed tiled events (tiles_before > 0, a new n_long)
        assert any(done[i] > done[0] for i in np.flatnonzero(spine))
        tiled_chunks = sorted(set(done[tiled].tolist()))
        assert len(tiled_chunks) >= 3
    chunks = sc.long_chunks(n)
    assert sc.streams(n, chunks[-2]) and n - sc.rounded(chunks[-2]) * (sc.chunk_count(n, chunks[-2]) - 1) < sc.K1_TILE
    assert not sc.streams(n, chunks[-1])
    assert all(sc.streams(n, c) for c in chunks[:-1])


def test_edge_trace_places_crossings_and_non_finite_samples_on_chunk_boundaries():
    case = sc.cases()["edges_mask7"]
    x, n, C = case.current(), case.n, sc.EDGE_CHUNK
    for chunk in case.chunks:
        assert C % sc.rounded(chunk) == 0 and sc.streams(n, chunk)
    assert n % C == 1                                                  # a final chunk of one sample
    runs, ws, wl = selected(case)
    start, length, mn, mx, below = runs
    starts = set(start.tolist())
    assert {C, 2 * C + 1, 3 * C - 1} <= set(ws.tolist())                # crossings at b, b + 1, b - 1
    assert 4 * C in set((ws + wl).tolist())                            # an event whose last sample is b - 1
    assert ws[-1] + wl[-1] == n and ws[-1] < 12 * C                    # the open last event, finished by 1 sample
    for b, inside in ((5 * C, True), (6 * C, True), (7 * C, False), (8 * C, False)):
        assert not np.isfinite(x[b - 1]) and not np.isfinite(x[b])
        assert (x[b - 2] < 110) == inside and (x[b + 1] < 110) == inside
    assert np.isnan(x[5 * C - 1]) and np.isposinf(x[5 * C]) and 5 * C - 1 in starts      # NaN / +inf split the event
    assert np.isneginf(x[6 * C - 1]) and np.isneginf(x[6 * C])
    r = np.searchsorted(start, 6 * C - 1, side="right") - 1
    assert below[r] and start[r] < 6 * C - 1 and start[r] + length[r] > 6 * C and mn[r] == -np.inf
    for b, which in ((9 * C, mn), (10 * C, mx), (11 * C, mx)):         # run extrema on the first sample of a chunk
        r = np.searchsorted(start, b, side="right") - 1
        assert start[r] < b and which[r] == x[b]
    assert np.isnan(x[7 * C - 1]) and np.isneginf(x[7 * C]) and np.isposinf(x[8 * C - 1]) and np.isnan(x[8 * C])
    # with every run an event the NaN-bearing open-channel runs are events too
    _, ws0, _ = selected(sc.cases()["edges_mask0"])
    assert len(ws0) == len(start)


def test_dense_trace_completes_more_than_1024_runs_in_a_chunk_from_an_odd_offset():
    case = sc.cases()["dense"]
    n = case.n
    runs, ws, wl = selected(case)
    start, length = runs[0], runs[1]
    assert len(start) <= n // 256 + 4096                               # no run-table overflow
    for chunk in case.chunks:
        done = sc.completions(n, chunk, start, length)
        per = np.bincount(done, minlength=sc.chunk_count(n, chunk))
        before = np.concatenate(([0], np.cumsum(per)[:-1]))
        assert any(per[k] > sc.SEL_THREADS and before[k] % sc.SEL_THREADS for k in range(len(per))), chunk
    assert len(ws) == 1400 and sc.streams(n, case.chunks[0])


def test_overflow_trace_exceeds_the_streamed_run_table():
    x = sc.overflow_trace()
    runs = sc.oracle.threshold_runs(x.astype(np.float64), 110.0)
    assert len(runs[0]) > len(x) // 256 + 4096 and sc.streams(len(x), 1 << 18)


def test_rule_sets_select_above_threshold_runs_non_finite_runs_and_exact_limits():
    sets = sc.rule_sets()
    cases = sc.cases()
    x = sc.rule_trace()
    n = len(x)
    got = {name: selected(cases["rules_" + name]) for name in sets}
    runs = got["mask0"][0]
    start, length, mn, mx, below = runs
    assert not below[0] and not below[-1]                              # the trace starts and ends above
    nan_run = int(np.flatnonzero(np.isnan(mn))[0])
    assert not below[nan_run]
    masks = {sets[k]["rule_mask"] for k in sets}
    assert masks == {0, 1, 2, 4, 9, 7, 15}
    for name, (_, ws, wl) in got.items():
        s = set(ws.tolist())
        above_selected = any(not below[np.searchsorted(start, v)] for v in s)
        if name in ("mask0", "mask1_1000", "mask2_all"):
            assert 0 in s and start[-1] in s and above_selected, name  # run at sample 0 and the open last run
        if name in ("mask0", "mask1_1000"):
            assert start[nan_run] in s, name                           # duration-only rules accept NaN runs
        if name in ("mask2_all", "mask2_at_min", "mask4", "mask7", "mask15"):
            assert start[nan_run] not in s, name                       # min / max rules reject them
        if name in ("mask4", "mask7", "mask15"):
            assert not above_selected, name
    for cname in cases:
        if cname.startswith("rules_"):
            assert all(sc.streams(n, c) for c in cases[cname].chunks)
    # duration limits at an actual event length L and L +- 1 (strict comparisons)
    ev = np.flatnonzero(below)
    L = int(length[ev[7]])
    assert sets["mask1_at_len+0"]["duration_gt"] == L
    hit = lambda name: start[ev[7]] in set(got[name][1].tolist())
    assert hit("mask1_at_len-1") and not hit("mask1_at_len+0") and not hit("mask1_at_len+1")
    assert hit("mask9_at_len+1") and not hit("mask9_at_len+0") and not hit("mask9_at_len-1")
    m = mn[ev[11]]
    assert sets["mask2_at_min"]["min_gt"] == m
    assert start[ev[11]] not in set(got["mask2_at_min"][1].tolist())
    assert start[ev[11]] in set(got["mask2_all"][1].tolist())


@pytest.mark.parametrize("name", sorted(sc.ADC_SOURCES))
def test_adc_cases_put_int16_extremes_on_chunk_edges(name):
    case = sc.cases()[name]
    c = case.x.counts
    for k in (3, 7, 11, 19):
        b = k * sc.EDGE_CHUNK
        assert c[b - 1] == -32768 and c[b] == 32767
    assert all(sc.streams(case.n, ch) for ch in case.chunks)
    _, ws, wl = selected(case)
    assert (wl > sc.K2F_MAX_LEN).sum() >= 6


def test_every_streamed_case_streams_and_the_big_trace_spans_two_default_chunks():
    for name, case in sc.cases().items():
        assert any(sc.streams(case.n, c) for c in case.chunks), name
    x = sc.big_trace()
    n = len(x)
    assert 17 << 20 > n - (1 << 20) and n <= 19000000 and sc.streams(n, 0) and sc.chunk_count(n, 0) == 2
    runs = sc.oracle.threshold_runs(x.astype(np.float64), 110.0)
    keep = sc.oracle.select_runs(x.astype(np.float64), runs, sc.rule_lambdas(sc.RULES7))
    ws, wl = runs[0][keep], runs[1][keep]
    D = sc.DEFAULT_CHUNK
    assert any((s < D) and (s + l > D) and l > sc.K2F_MAX_LEN for s, l in zip(ws, wl))
    assert ws[-1] + wl[-1] == n and wl[-1] > sc.K2F_MAX_LEN and len(ws) == 62
