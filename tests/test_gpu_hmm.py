"""HMM decoding on the device (csrc/hmm.cuh) against the NumPy oracle, run on the device's own segment means.

Viterbi must be bit-equal (log-probability and path), forward within 1e-10 * (1 + |logp|).  The merge must give the
boundaries oracle.hmm.hmm_merge gives for the device's states, with statistics within the usual parity bars, on every
sample source."""
import ctypes

import numpy as np
import pytest

import oracle
from oracle import hmm as hmm_oracle
from pypore_b200 import _lib, synth
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import File
from pypore_b200.hmm import HMM
from pypore_b200.parsers import RuleSet, SpeedyStatSplit, lambda_event_parser

pytestmark = pytest.mark.gpu

RULES = RuleSet(duration_gt=1000, min_gt=-0.5, max_lt=110)
FS = 1e5
GAINS = {"default": dict(min_width=100, window_width=10000),
         "psps10": dict(min_width=100, window_width=10000, prior_segments_per_second=10)}


def bits(v):
    return np.asarray(v, np.float64).tobytes()


def level_model(S, seed=0, spread=(0.0, 110.0), ends=False, dup=None):
    """S states spread over the trace's current levels, sticky transitions, some forbidden edges."""
    rng = np.random.default_rng(seed)
    mean = np.sort(rng.uniform(*spread, S))
    std = rng.uniform(1.0, 6.0, S)
    trans = rng.uniform(0.0, 1.0, (S, S)) + 4 * np.eye(S)
    trans[rng.uniform(size=(S, S)) < 0.2] = 0.0
    np.fill_diagonal(trans, 4.0)
    starts = rng.uniform(0.1, 1.0, S)
    end = rng.uniform(0.0, 0.5, S) if ends else None
    if dup is not None:                   # state k copies state j: exact ties at every step
        j, k = dup
        mean[k], std[k], starts[k] = mean[j], std[j], starts[j]
        trans[k, :] = trans[j, :]     # same way out ...
        trans[:, k] = trans[:, j]     # ... and in
        if end is not None:
            end[k] = end[j]
    return HMM(mean, std, trans, starts=starts, ends=end)


def check_viterbi(model, seqs):
    got = model.viterbi_many(seqs)
    for q, (lp, st) in zip(seqs, got):
        olp, ost = hmm_oracle.hmm_viterbi(q, **model.params())
        assert bits(lp) == bits(olp), (lp, olp)
        assert np.array_equal(st, ost)
    return got


def check_forward(model, seqs):
    got = model.log_probability_many(seqs)
    worst = 0.0
    for q, lp in zip(seqs, got):
        olp = hmm_oracle.hmm_forward(q, **model.params())
        if not np.isfinite(olp):
            assert bits(lp) == bits(olp), (lp, olp)
            continue
        err = abs(lp - olp) / (1 + abs(olp))
        worst = max(worst, err)
        assert err <= 1e-10, (lp, olp)
    return worst


def parse_file(x, gain="psps10", hmm=None, filter_params=None, timestep=1000. / FS):
    f = File(current=x, timestep=timestep)
    f.parse(parser=lambda_event_parser(threshold=110, rules=RULES), segmenter=SpeedyStatSplit(**GAINS[gain]),
            filter_params=filter_params, hmm=hmm)
    return f


def event_means(table, n_events):
    b = np.searchsorted(table["event"], np.arange(n_events + 1))
    return [table["mean"][b[i]:b[i + 1]] for i in range(n_events)]


@pytest.fixture(scope="module")
def tier_a():
    x = synth.make_trace(500, seed=0, tier="A")   # c1 size: 500 events, ~6 M samples
    return x


@pytest.mark.parametrize("S", [1, 2, 31, 32, 33, 64, 127, 128])
def test_viterbi_and_forward_equal_the_oracle_on_device_means(tier_a, S):
    f = parse_file(tier_a)
    seqs = event_means(f.segment_table, len(f.event_table["start"]))
    model = level_model(S, seed=S, ends=S % 2 == 0)
    check_viterbi(model, seqs)
    check_forward(model, seqs)


@pytest.mark.parametrize("gain", sorted(GAINS))
def test_tier_a_traces_at_both_gains(tier_a, gain):
    f = parse_file(tier_a, gain=gain)
    seqs = event_means(f.segment_table, len(f.event_table["start"]))
    for S in (8, 40):
        check_viterbi(level_model(S, seed=7), seqs)


@pytest.mark.parametrize("S,dup", [(2, (0, 1)), (16, (3, 9)), (64, (10, 50)), (128, (0, 127))])
def test_duplicate_states_tie_to_the_lowest_index(S, dup):
    rng = np.random.default_rng(S)
    model = level_model(S, seed=S, dup=dup)
    seqs = [rng.choice(model.mean, n) + rng.normal(0, 2, n) for n in (1, 2, 17, 300)]
    got = check_viterbi(model, seqs)
    assert not any((st == dup[1]).any() for _, st in got)   # the higher duplicate never wins a tie


@pytest.mark.parametrize("S", [3, 32, 33, 128])
def test_forbidden_impossible_nan_and_single_value_sequences(S):
    rng = np.random.default_rng(5)
    mean = np.linspace(0, 100, S)
    trans = np.eye(S) + np.eye(S, k=1)          # left to right only
    starts = np.zeros(S)
    starts[0] = 1
    ends = np.zeros(S)
    ends[-1] = 1
    model = HMM(mean, np.full(S, 2.0), trans, starts=starts, ends=ends)
    ramp = np.repeat(mean, 3) + rng.normal(0, 0.5, 3 * S)
    seqs = [ramp, ramp[::-1], np.array([50.0]), np.array([mean[-1]]), np.r_[ramp[:5], np.nan, ramp[5:]],
            np.array([np.inf, 1.0]), np.array([-np.inf]), ramp[:2]]
    got = check_viterbi(model, seqs)
    assert got[0][0] > -np.inf and got[0][1][0] == 0 and got[0][1][-1] == S - 1
    for k in (2, 3, 4, 5, 6, 7):                 # too short to reach the end state, NaN, +-inf: states -1
        assert (got[k][1] == -1).all()
    assert np.isnan(got[4][0]) and got[2][0] == got[5][0] == -np.inf
    check_forward(model, seqs)
    open_model = HMM(mean, np.full(S, 2.0), trans)   # without ends a single value is possible
    check_viterbi(open_model, [np.array([50.0]), np.array([mean[0]])])


def test_long_sequences_forward_error_stays_within_the_bar():
    rng = np.random.default_rng(11)
    for S in (8, 128):
        model = level_model(S, seed=3)
        q = rng.choice(model.mean, 100_000) + rng.normal(0, 3, 100_000)
        assert check_forward(model, [q]) <= 1e-10
        check_viterbi(model, [q])


def test_one_million_sample_event_at_default_gain():
    x = synth.make_long_event(1_000_000, seed=100, tier="A").astype(np.float64)
    segs = SpeedyStatSplit(**GAINS["default"]).parse(x)
    assert len(segs) > 1000
    means = np.array([s.mean for s in segs])
    for S in (4, 32, 96):
        check_viterbi(level_model(S, seed=S), [means])


def test_resident_decode_equals_host_sequences(ctx, tier_a):
    f = parse_file(tier_a, hmm=None)
    mw, MW, W, gain = SpeedyStatSplit(**GAINS["psps10"])._params()
    counts = ctx.pipeline(110, rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0, min_width=mw,
                          max_width=MW, window_width=W, min_gain=gain, host_trace=np.asarray(tier_a, np.float32))
    n_ev, n_seg = counts["events"], counts["segments"]
    tab = ctx.segments(n_seg)
    seqs = event_means(tab, n_ev)
    for S in (5, 32, 100):
        model = level_model(S, seed=S, ends=True)
        for algorithm in ("viterbi", "forward"):
            assert ctx.hmm_decode(model, algorithm) == n_seg
            lp, st = ctx.hmm_download(n_ev, n_seg if algorithm == "viterbi" else None)
            ctx.hmm_decode_sequences(model, algorithm, seqs)
            lp2, st2 = ctx.hmm_download(n_ev, n_seg if algorithm == "viterbi" else None)
            assert bits(lp) == bits(lp2)
            if algorithm == "viterbi":
                assert np.array_equal(st, st2)
    assert np.array_equal(tab["start"], f.segment_table["start"])


def test_refusals():
    c = _lib.Context(0)
    try:
        model = level_model(4)
        with pytest.raises(_lib.PyPoreCudaError, match="-4"):     # PP_ERR_STATE: no resident statistics
            c.hmm_decode(model)
        with pytest.raises(_lib.PyPoreCudaError, match="-4"):     # nothing decoded yet
            c.hmm_download(1)
        c.upload_events_f64([np.r_[np.zeros(500), np.ones(500)]])
        c.statsplit(100, 1000000, 10000, 0.0)
        with pytest.raises(_lib.PyPoreCudaError, match="-4"):     # split, but no statistics
            c.hmm_decode(model)
        c.segment_stats()
        with pytest.raises(ValueError):                            # PP_ERR_ARG: merge with forward
            c.hmm_decode(model, "forward", merge=True)
        for S in (0, 129):
            m = c._hmm(model)
            m.n_states = S
            n = ctypes.c_int64()
            assert c._L.pp_hmm_decode(c._h, ctypes.byref(m), 0, 0, ctypes.byref(n)) == _lib.PP_ERR_ARG
            assert c._L.pp_hmm_decode_sequences(c._h, ctypes.byref(m), 0, None, None, 0) == _lib.PP_ERR_ARG
        with pytest.raises(ValueError):                            # empty sequence
            c.hmm_decode_sequences(model, "viterbi", [np.zeros(3), np.zeros(0)])
        n = c.hmm_decode(model, "forward")
        with pytest.raises(_lib.PyPoreCudaError, match="-4"):     # forward computes no states
            c.hmm_download(1, n)
        assert c.hmm_download(1)[0].shape == (1,)
    finally:
        c.close()


def adc_of(x32, scale=1.0 / 32, offset=0.0):
    return AdcTrace(np.round((x32.astype(np.float64) - offset) / scale).astype(np.int16), scale, offset)


def sources(x):
    x32 = np.asarray(x, np.float32)
    x64 = x32.astype(np.float64) + 1e-7          # not float32-representable: stays float64 on the device
    return {"float32": (x32, x32.astype(np.float64)), "float64": (x64, x64),
            "adc": (adc_of(x32, 0.0305, 0.0123), adc_of(x32, 0.0305, 0.0123).decode())}


@pytest.mark.parametrize("source", ["float32", "float64", "adc"])
@pytest.mark.parametrize("filt", [None, (1, 2000)])
def test_file_parse_merge_matches_the_oracle(source, filt):
    x = synth.make_trace(60, seed=3, tier="A")
    trace, decoded = sources(x)[source]
    model = level_model(6, seed=2)
    plain = parse_file(trace, filter_params=filt)
    merged = parse_file(trace, filter_params=filt, hmm=model)
    assert "state" not in plain.segment_table and "log_probability" not in plain.event_table
    n_ev = len(plain.event_table["start"])
    assert n_ev > 10
    pt, mt = plain.segment_table, merged.segment_table
    text = merged.to_json()                       # the reference's format: the new columns are not written
    assert '"state"' not in text and '"log_probability"' not in text
    seqs = event_means(pt, n_ev)
    got = model.viterbi_many(seqs)
    states = np.concatenate([st for _, st in got])
    assert bits(merged.event_table["log_probability"]) == bits([lp for lp, _ in got])
    e, s, t, q = hmm_oracle.hmm_merge(pt["event"], pt["start"], pt["end"], states)
    assert len(e) < len(pt["event"])
    for name, want in (("event", e), ("start", s), ("end", t), ("state", q)):
        assert np.array_equal(mt[name], want), name
    for i in range(n_ev):
        ev = merged.events[i]
        a, n = int(merged.event_table["start"][i]), int(merged.event_table["length"][i])
        samples = ev.current if filt is not None else decoded[a:a + n]
        sel = mt["event"] == i
        m, sd, mn, mx = oracle.segment_stats(np.asarray(samples, np.float64), mt["start"][sel], mt["end"][sel])
        assert np.allclose(mt["mean"][sel], m, rtol=1e-9, atol=1e-12)
        assert np.allclose(mt["std"][sel], sd, rtol=1e-9, atol=1e-12)
        assert np.array_equal(mt["min"][sel], mn) and np.array_equal(mt["max"][sel], mx)
        assert [seg.state for seg in ev.segments] == list(mt["state"][sel])


def test_event_parse_with_hmm_equals_file_parse():
    x = synth.make_trace(40, seed=4, tier="A").astype(np.float64) + 1e-7
    model = level_model(6, seed=2)
    f = parse_file(x, hmm=model)
    mt = f.segment_table
    g = parse_file(x)
    for i, ev in enumerate(g.events):
        n = ev.parse(parser=SpeedyStatSplit(**GAINS["psps10"]), hmm=model)
        sel = mt["event"] == i
        assert n == int(sel.sum())
        assert [s.start for s in ev.segments] == list(mt["start"][sel] / f.second)
        assert [s.state for s in ev.segments] == list(mt["state"][sel])
        assert np.allclose([s.mean for s in ev.segments], mt["mean"][sel], rtol=1e-12, atol=0)
        assert bits(ev.log_probability) == bits(f.event_table["log_probability"][i])


def test_apply_hmm_decodes_the_segment_means():
    x = synth.make_trace(10, seed=6, tier="A").astype(np.float64)
    f = parse_file(x)
    model = level_model(5, seed=9)
    ev = f.events[0]
    means = np.array([s.mean for s in ev.segments])
    lp, st = ev.apply_hmm(model)
    olp, ost = hmm_oracle.hmm_viterbi(means, **model.params())
    assert bits(lp) == bits(olp) and np.array_equal(st, ost)
    assert abs(ev.apply_hmm(model, "forward") - hmm_oracle.hmm_forward(means, **model.params())) <= 1e-10 * (1 + abs(olp))
    with pytest.raises(ValueError):
        ev.apply_hmm(model, "posterior")
