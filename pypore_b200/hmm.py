"""Hidden Markov models over segment means, decoded on the device (csrc/hmm.cuh).

What PyPore's segment tables are for: ``Event.apply_hmm`` / ``Event.parse(parser, hmm)`` (reference
DataTypes.py:292-355) hand the segment means of an event to a yahmm model.  ``HMM`` is that model for the common
case -- S <= 128 emitting states with normal emissions, a transition matrix, start and optional end
probabilities -- with these semantics:

* the host normalises each row of ``transitions`` (together with ``ends[i]`` when ``ends`` is given) and ``starts``
  (default uniform), and takes every log once in NumPy float64 (0 -> -inf);
* emission e_j(x) = c_j - 0.5 * (z * z), z = (x - mean_j) * r_j, r_j = 1 / std_j, c_j = -log(std_j) - log(2 pi) / 2;
* Viterbi: the best path and its log-probability, bit-equal to ``oracle.hmm.hmm_viterbi``; ties go to the lowest state
  index.  A NaN value gives log-probability NaN, an impossible sequence -inf; both give every state -1;
* forward: the log-likelihood, within 1e-10 * (1 + |logp|) of the exact value (CUDA exp / log).

Silent states other than the end term, pseudo-counts, edge tying and posteriors are not modelled.
"""
import numpy as np

from . import _lib

MAX_STATES = 128


def _vector(v, n, what):
    a = np.array(v, dtype=np.float64).reshape(-1)
    if a.shape[0] != n:
        raise ValueError("%s must have %d entries, got %d" % (what, n, a.shape[0]))
    return a


def _nonnegative(a, what):
    if not np.all(np.isfinite(a)) or np.any(a < 0):
        raise ValueError("%s must be finite and non-negative" % what)


class HMM(object):
    """``HMM(means, stds, transitions, starts=None, ends=None, names=None)``: S normal-emission states.

    ``transitions[i][j]`` is the weight of i -> j, ``ends[i]`` that of leaving the model from i; rows are
    normalised (with the end weight), as are ``starts``.  The log-space arrays the device uses are attributes:
    ``mean``, ``inv_std``, ``log_norm``, ``log_start``, ``log_trans`` (S x S, row = predecessor), ``log_end``
    (None without ``ends``)."""

    def __init__(self, means, stds, transitions, starts=None, ends=None, names=None):
        mean = np.array(means, dtype=np.float64).reshape(-1)
        S = mean.shape[0]
        if not 1 <= S <= MAX_STATES:
            raise ValueError("an HMM has 1..%d states, got %d" % (MAX_STATES, S))
        std = _vector(stds, S, "stds")
        if not np.all(np.isfinite(mean)) or not np.all(np.isfinite(std)) or np.any(~(std > 0)):
            raise ValueError("means and stds must be finite, stds > 0")
        trans = np.array(transitions, dtype=np.float64)
        if trans.shape != (S, S):
            raise ValueError("transitions must be %d x %d, got %s" % (S, S, trans.shape))
        _nonnegative(trans, "transitions")
        start = np.ones(S) if starts is None else _vector(starts, S, "starts")
        _nonnegative(start, "starts")
        end = None if ends is None else _vector(ends, S, "ends")
        if end is not None:
            _nonnegative(end, "ends")
        rows = trans.sum(axis=1) + (end if end is not None else 0.0)
        if np.any(rows == 0):
            raise ValueError("transition rows %s sum to 0" % np.flatnonzero(rows == 0).tolist())
        if start.sum() == 0:
            raise ValueError("starts sum to 0")
        self.names = list(names) if names is not None else ["s%d" % j for j in range(S)]
        if len(self.names) != S:
            raise ValueError("names must have %d entries" % S)
        self.n_states = S
        self.transitions = trans / rows[:, None]
        self.starts = start / start.sum()
        self.ends = end / rows if end is not None else None
        with np.errstate(divide="ignore"):
            self.log_trans = np.ascontiguousarray(np.log(self.transitions))
            self.log_start = np.log(self.starts)
            self.log_end = np.log(self.ends) if end is not None else None
        self.mean = mean
        self.std = std
        self.inv_std = 1.0 / std
        self.log_norm = -np.log(std) - 0.5 * np.log(2 * np.pi)

    def params(self):
        """The log-space model as keyword arguments of oracle.hmm.hmm_viterbi / hmm_forward."""
        return dict(mean=self.mean, inv_std=self.inv_std, log_norm=self.log_norm, log_start=self.log_start,
                    log_trans=self.log_trans, log_end=self.log_end)

    @staticmethod
    def _sequences(seqs):
        out = [np.ascontiguousarray(np.asarray(q, dtype=np.float64).reshape(-1)) for q in seqs]
        if any(q.shape[0] == 0 for q in out):
            raise ValueError("cannot decode an empty sequence")
        return out

    def viterbi_many(self, seqs, context=None):
        """[(log-probability, states int32 array)] of every sequence, decoded in one device call."""
        seqs = self._sequences(seqs)
        ctx = context or _lib.default_context()
        lens = ctx.hmm_decode_sequences(self, "viterbi", seqs)
        logp, states = ctx.hmm_download(len(seqs), int(lens.sum()))
        return list(zip(logp.tolist(), np.split(states, np.cumsum(lens)[:-1]))) if len(seqs) else []

    def log_probability_many(self, seqs, context=None):
        """Forward log-likelihood of every sequence (float64 array), in one device call."""
        seqs = self._sequences(seqs)
        ctx = context or _lib.default_context()
        ctx.hmm_decode_sequences(self, "forward", seqs)
        return ctx.hmm_download(len(seqs))[0]

    def viterbi(self, seq):
        """(log-probability of the best path, its states)."""
        return self.viterbi_many([seq])[0]

    def log_probability(self, seq):
        """Forward log-likelihood of one sequence."""
        return float(self.log_probability_many([seq])[0])
