"""HMM decoding without a GPU: the NumPy oracle against brute-force enumeration of every path, the model's
validation and normalisation, and the segment merge on hand-made state sequences."""
import itertools
import math

import numpy as np
import pytest

from oracle import hmm as hmm_oracle
from pypore_b200.hmm import HMM


def random_model(rng):
    """A small model with the awkward cases mixed in: duplicate states (exact ties), zero transitions and starts,
    ends present or absent."""
    S = int(rng.integers(1, 5))
    mean = rng.normal(0.0, 2.0, S)
    std = rng.uniform(0.3, 2.0, S)
    trans = rng.uniform(0.0, 1.0, (S, S))
    trans[rng.uniform(size=(S, S)) < 0.3] = 0.0
    starts = rng.uniform(0.0, 1.0, S)
    starts[rng.uniform(size=S) < 0.3] = 0.0
    ends = rng.uniform(0.0, 1.0, S) if rng.uniform() < 0.5 else None
    if S > 1 and rng.uniform() < 0.5:   # state k duplicates state j: same emission, start, incoming edges, end
        j, k = rng.choice(S, 2, replace=False)
        mean[k], std[k], starts[k], trans[:, k] = mean[j], std[j], starts[j], trans[:, j]
        if ends is not None:
            ends[k] = ends[j]
    for i in range(S):              # no row may sum to 0
        if trans[i].sum() == 0 and (ends is None or ends[i] == 0):
            trans[i, rng.integers(S)] = 1.0
    if starts.sum() == 0:
        starts[rng.integers(S)] = 1.0
    return HMM(mean, std, trans, starts=starts, ends=ends)


def random_sequence(rng, model):
    T = int(rng.integers(1, 7))
    x = rng.choice(model.mean, T) + rng.normal(0.0, 0.5, T)
    u = rng.uniform()
    if u < 0.1:
        x[rng.integers(T)] = np.nan
    elif u < 0.2:
        x[rng.integers(T)] = np.inf
    elif u < 0.3:
        x[rng.integers(T)] = -np.inf
    return x


def brute_force(x, p):
    """Every path's score in Python floats (one rounding per operation, the device's order); delta_t(j) as the max over
    all prefixes ending in j; the path by the traceback rule (lowest index among the maxima) over those deltas."""
    S, T = len(p["mean"]), len(x)
    lend = p["log_end"] if p["log_end"] is not None else np.zeros(S)
    A = p["log_trans"]

    def e(t, j):
        z = (float(x[t]) - float(p["mean"][j])) * float(p["inv_std"][j])
        return float(p["log_norm"][j]) - 0.5 * (z * z)

    delta = [[-math.inf] * S for _ in range(T)]
    finals = []
    for path in itertools.product(range(S), repeat=T):
        s = float(p["log_start"][path[0]]) + e(0, path[0])
        delta[0][path[0]] = max(delta[0][path[0]], s)
        for t in range(1, T):
            s = (s + float(A[path[t - 1], path[t]])) + e(t, path[t])
            delta[t][path[t]] = max(delta[t][path[t]], s)
        finals.append(s + float(lend[path[-1]]))
    logp = max(finals)
    M = logp
    fwd = -math.inf if M == -math.inf else M + math.log(math.fsum(math.exp(f - M) for f in finals))
    if logp == -math.inf:
        return logp, np.full(T, -1, np.int32), fwd
    last = [delta[T - 1][j] + float(lend[j]) for j in range(S)]
    j = last.index(max(last))
    states = [j]
    for t in range(T - 1, 0, -1):
        v = [delta[t - 1][i] + float(A[i, j]) for i in range(S)]
        j = v.index(max(v))
        states.append(j)
    return logp, np.array(states[::-1], np.int32), fwd


def test_oracle_matches_brute_force_on_seeded_models():
    rng = np.random.default_rng(2024)
    seen = dict(tie=0, zero=0, ends=0, no_ends=0, nan=0, inf=0, t1=0, impossible=0)
    for case in range(400):
        model = random_model(rng)
        p = model.params()
        x = random_sequence(rng, model)
        logp, states = hmm_oracle.hmm_viterbi(x, **p)
        fwd = hmm_oracle.hmm_forward(x, **p)
        seen["ends" if p["log_end"] is not None else "no_ends"] += 1
        seen["t1"] += len(x) == 1
        seen["zero"] += bool(np.isinf(p["log_trans"]).any() or np.isinf(p["log_start"]).any())
        seen["inf"] += bool(np.isinf(x).any())
        if np.isnan(x).any():
            seen["nan"] += 1
            assert math.isnan(logp) and math.isnan(fwd) and (states == -1).all()
            continue
        bl, bs, bf = brute_force(x, p)
        assert np.float64(logp).tobytes() == np.float64(bl).tobytes(), case
        assert np.array_equal(states, bs), (case, states, bs)
        if bl == -math.inf:
            seen["impossible"] += 1
            assert fwd == -math.inf and (states == -1).all()
        else:
            assert abs(fwd - bf) <= 1e-13 * (1 + abs(bf)), (case, fwd, bf)
            # an exact tie between two states at some step
            S = len(p["mean"])
            if S > 1 and len(set(map(float, p["mean"]))) < S:
                seen["tie"] += 1
    assert all(v > 0 for v in seen.values()), seen


def test_viterbi_ties_go_to_the_lowest_index():
    # two identical states: every step ties, so the path is state 0 throughout
    m = HMM([0.0, 0.0], [1.0, 1.0], [[1, 1], [1, 1]])
    logp, states = hmm_oracle.hmm_viterbi([0.1, -0.3, 0.2], **m.params())
    assert (states == 0).all()
    # a third state duplicating state 1 behind a distinct state 0
    m = HMM([5.0, 0.0, 0.0], [1.0, 1.0, 1.0], [[1, 1, 1]] * 3)
    assert hmm_oracle.hmm_viterbi([0.0, 5.0, 0.0], **m.params())[1].tolist() == [1, 0, 1]


def test_forbidden_transitions_make_a_sequence_impossible():
    m = HMM([0.0, 10.0], [1.0, 1.0], [[1, 0], [0, 1]], starts=[1, 0])
    logp, states = hmm_oracle.hmm_viterbi([0.0, 10.0], **m.params())
    assert logp > -np.inf and states.tolist() == [0, 0]
    m = HMM([0.0, 10.0], [1.0, 1.0], [[1, 0], [0, 1]], starts=[1, 0], ends=[0, 1])
    logp, states = hmm_oracle.hmm_viterbi([0.0, 10.0], **m.params())
    assert logp == -np.inf and (states == -1).all()
    assert hmm_oracle.hmm_forward([0.0, 10.0], **m.params()) == -np.inf


def test_hmm_normalises_rows_with_their_end_weight_and_the_starts():
    m = HMM([0, 1, 2], [1, 2, 3], [[1, 1, 2], [0, 3, 0], [1, 0, 0]], starts=[2, 0, 2], ends=[0, 1, 3])
    assert np.allclose(m.transitions.sum(axis=1) + m.ends, 1.0, rtol=0, atol=1e-15)
    assert np.array_equal(m.transitions[0], [0.25, 0.25, 0.5]) and np.array_equal(m.ends, [0.0, 0.25, 0.75])
    assert np.array_equal(m.starts, [0.5, 0.0, 0.5])
    assert m.log_start[1] == -np.inf and m.log_trans[1, 0] == -np.inf and m.log_end[0] == -np.inf
    with np.errstate(divide="ignore"):
        assert np.array_equal(m.log_trans, np.log(m.transitions))
    assert np.array_equal(m.inv_std, 1.0 / np.array([1.0, 2.0, 3.0]))
    assert np.array_equal(m.log_norm, -np.log([1.0, 2.0, 3.0]) - 0.5 * np.log(2 * np.pi))
    u = HMM([0, 1], [1, 1], [[1, 3], [1, 1]])
    assert np.array_equal(u.starts, [0.5, 0.5]) and u.log_end is None
    assert np.array_equal(u.transitions, [[0.25, 0.75], [0.5, 0.5]])


@pytest.mark.parametrize("kwargs", [
    dict(means=[0] * 129, stds=[1] * 129, transitions=np.ones((129, 129))),
    dict(means=[], stds=[], transitions=np.ones((0, 0))),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 0], [0, 0]]),                          # a row sums to 0
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1], [1, 1]], starts=[0, 0]),           # starts sum to 0
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, -1], [1, 1]]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, np.nan], [1, 1]]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, np.inf], [1, 1]]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1], [1, 1]], starts=[1, -1]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1], [1, 1]], starts=[1, np.nan]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1], [1, 1]], ends=[np.inf, 0]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1], [1, 1]], ends=[-1, 0]),
    dict(means=[0, np.nan], stds=[1, 1], transitions=[[1, 1], [1, 1]]),
    dict(means=[0, np.inf], stds=[1, 1], transitions=[[1, 1], [1, 1]]),
    dict(means=[0, 1], stds=[1, 0], transitions=[[1, 1], [1, 1]]),
    dict(means=[0, 1], stds=[1, -2], transitions=[[1, 1], [1, 1]]),
    dict(means=[0, 1], stds=[1, 1], transitions=[[1, 1, 1], [1, 1, 1]]),
    dict(means=[0, 1], stds=[1], transitions=[[1, 1], [1, 1]]),
])
def test_hmm_rejects_invalid_models(kwargs):
    with pytest.raises(ValueError):
        HMM(**kwargs)


def test_hmm_accepts_128_states_and_a_zero_row_with_an_end():
    HMM(np.arange(128.0), np.ones(128), np.ones((128, 128)))
    m = HMM([0, 1], [1, 1], [[1, 1], [0, 0]], ends=[0, 1])
    assert np.array_equal(m.ends, [0, 1]) and (m.log_trans[1] == -np.inf).all()


def test_merge_joins_runs_of_one_state_within_an_event():
    event = np.array([0, 0, 0, 0, 1, 1, 1, 2, 2, 3])
    start = np.array([0, 10, 20, 30, 0, 5, 9, 0, 4, 0])
    end = np.array([10, 20, 30, 40, 5, 9, 12, 4, 8, 7])
    state = np.array([1, 1, 2, 1, 1, 1, 1, -1, -1, 0])
    e, s, t, q = hmm_oracle.hmm_merge(event, start, end, state)
    assert e.tolist() == [0, 0, 0, 1, 2, 2, 3]
    assert s.tolist() == [0, 20, 30, 0, 0, 4, 0]
    assert t.tolist() == [20, 30, 40, 12, 4, 8, 7]
    assert q.tolist() == [1, 2, 1, 1, -1, -1, 0]
    # the same state at the end of one event and the start of the next does not join them
    e, s, t, q = hmm_oracle.hmm_merge([0, 1], [0, 0], [3, 4], [2, 2])
    assert e.tolist() == [0, 1] and t.tolist() == [3, 4]
    e, s, t, q = hmm_oracle.hmm_merge(np.zeros(0, int), np.zeros(0, int), np.zeros(0, int), np.zeros(0, int))
    assert len(e) == 0
