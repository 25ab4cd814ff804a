"""NumPy restatement of HMM decoding over segment means (TEST INFRASTRUCTURE, see oracle/__init__.py).

The model is given in log space, as pypore_b200.hmm.HMM.params() returns it: mean, inv_std = 1/sigma,
log_norm = -log(sigma) - log(2 pi)/2, log_start, log_trans [i, j] (i = predecessor), log_end (None: no end term).
Every operation below is one NumPy elementwise IEEE operation, in the order the device performs it.
"""
import numpy as np


def hmm_emission(x, mean, inv_std, log_norm):
    """e_j(x) = c_j - 0.5 * (z * z), z = (x - mu_j) * r_j."""
    z = (x - mean) * inv_std
    return log_norm - 0.5 * (z * z)


def _prepare(x, log_end, S):
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    if x.shape[0] == 0:
        raise ValueError("empty sequence")
    return x, np.zeros(S) if log_end is None else np.asarray(log_end, np.float64)


def hmm_viterbi(x, mean, inv_std, log_norm, log_start, log_trans, log_end=None):
    """(logp, states int32): delta_1 = log_start + e(x_1); delta_t(j) = max_i fl(delta_{t-1}(i) + logA_ij) + e_j(x_t)
    with the lowest i on ties; logp = max_j fl(delta_T(j) + log_end_j), lowest j on ties.  NaN anywhere in x: logp NaN;
    logp -inf: impossible; both give every state -1."""
    S = len(mean)
    x, lend = _prepare(x, log_end, S)
    T = x.shape[0]
    if np.isnan(x).any():
        return float("nan"), np.full(T, -1, np.int32)
    bp = np.zeros((T, S), np.int64)
    d = log_start + hmm_emission(x[0], mean, inv_std, log_norm)
    for t in range(1, T):
        v = d[:, None] + log_trans              # v[i, j]
        bp[t] = np.argmax(v, axis=0)            # first maximum: the lowest predecessor
        d = v[bp[t], np.arange(S)] + hmm_emission(x[t], mean, inv_std, log_norm)
    fin = d + lend
    j = int(np.argmax(fin))
    logp = float(fin[j])
    if logp == -np.inf:
        return logp, np.full(T, -1, np.int32)
    states = np.empty(T, np.int32)
    states[-1] = j
    for t in range(T - 1, 0, -1):
        j = int(bp[t, j])
        states[t - 1] = j
    return logp, states


def _logsumexp(v, axis):
    m = np.max(v, axis=axis)
    with np.errstate(invalid="ignore"):
        s = np.sum(np.exp(v - np.expand_dims(m, axis)), axis=axis)
    with np.errstate(divide="ignore"):
        return np.where(m == -np.inf, -np.inf, m + np.log(s))


def hmm_forward(x, mean, inv_std, log_norm, log_start, log_trans, log_end=None):
    """Forward log-likelihood: the Viterbi recursion with max replaced by m + log(sum_i exp(v_i - m)) (-inf when
    m = -inf).  NaN anywhere in x: NaN."""
    S = len(mean)
    x, lend = _prepare(x, log_end, S)
    if np.isnan(x).any():
        return float("nan")
    a = log_start + hmm_emission(x[0], mean, inv_std, log_norm)
    for t in range(1, x.shape[0]):
        a = _logsumexp(a[:, None] + log_trans, 0) + hmm_emission(x[t], mean, inv_std, log_norm)
    return float(_logsumexp(a + lend, 0))


def hmm_merge(event, start, end, state):
    """HMM-guided merge of a segment table (rows sorted by event, then start): every run of consecutive segments of
    one event that share a state >= 0 becomes one segment from the run's first start to its last end.  Returns
    (event, start, end, state) of the merged rows."""
    event, start, end, state = (np.asarray(a) for a in (event, start, end, state))
    n = event.shape[0]
    keep = np.ones(n, bool)
    if n > 1:
        keep[1:] = (event[1:] != event[:-1]) | (state[1:] < 0) | (state[1:] != state[:-1])
    first = np.flatnonzero(keep)
    last = np.append(first[1:], n)[:first.size] - 1
    return event[first], start[first], end[last], state[first]
