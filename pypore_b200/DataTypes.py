"""Container drivers behind the reference's names: ``File``, ``Event``, ``MetaEvent``, ``Experiment``, ``Sample``.

``File.parse(parser=...)``, ``Event.filter(order, cutoff)`` and ``Event.parse(parser=...)`` keep the reference's
signatures and side effects (DataTypes.py:258-289, 589-602).  The design is table-first:

* ``File.parse(..., segmenter=, filter_params=)`` runs threshold scan -> [Bessel filtfilt] -> split search ->
  statistics in ONE device-resident pass and keeps what came back as ``wire.FileTables`` (event rows, segment rows,
  in samples).  ``file.events`` is a lazy view on those tables: an ``Event`` / ``Segment`` object exists only once
  somebody indexes it.
* ``File.to_json`` / ``File.to_meta`` / the verbose lines of ``Experiment.parse`` work on the tables directly while
  no object has been handed out (``wire.file_tree``); after that they walk the objects, like the reference.

``File.parse(..., hmm=)`` and ``Event.parse(parser, hmm=)`` decode every event's segment means with a
``pypore_b200.hmm.HMM`` (Viterbi, on the device) and merge consecutive segments that share a state.  Plotting, MySQL
and .abf reading are out of scope (SURVEY.md section 2).
"""
import json
from functools import lru_cache

import numpy as np

from . import _lib, wire
from .adc import AdcTrace
from .core import MetaSegment, Segment
from .parsers import SpeedyStatSplit, lambda_event_parser, parser, _run_pipeline, _upload_trace

_STAT_SPAN = wire.FIELDS["MetaSegment"]


class MetaEvent(MetaSegment):
    """An event reduced to metadata (DataTypes.py:49-80): its segments are MetaSegments, no samples anywhere."""

    def to_json(self, filename=None):
        return wire.dumps(wire.expand_event(self, strict=False), filename)

    @classmethod
    def from_json(cls, _json):
        return cls(**json.loads(wire.source_text(_json)))

    from_segments = classmethod(lambda cls, segments: cls(segments=segments))
    n = property(lambda self: len(getattr(self, "segments", ())))

    def delete(self):
        self.__dict__.pop("state_parser", None)
        _each(self.segments, "delete")


def _each(items, method):
    """Call a no-argument method on every item."""
    for item in items:
        getattr(item, method)()


_NEEDS_CURRENT = "Cannot filter a metaevent. Must have the current."


def bessel_coefficients(order, cutoff, second):
    """(b, a, zi) for Event.filter: scipy.signal.bessel exactly as DataTypes.py:268-270
    requests it, plus the lfilter_zi steady state filtfilt starts from.  The design costs ~0.3 ms of
    Python per call and every event of every file of a batch asks for the same one: memoised (read-only arrays)."""
    return _bessel_coefficients(order, float(cutoff), float(second))


@lru_cache(maxsize=64)
def _bessel_coefficients(order, cutoff, second):
    from scipy import signal
    nyquist = second / 2.
    b, a = signal.bessel(order, cutoff / nyquist, btype='low', analog=0, output='ba')
    b = np.atleast_1d(np.asarray(b, np.float64))
    a = np.atleast_1d(np.asarray(a, np.float64))
    n = max(len(a), len(b))
    b = np.r_[b, np.zeros(n - len(b))] / a[0]
    a = np.r_[a, np.zeros(n - len(a))] / a[0]
    # lfilter_zi: solve (I - A^T) zi = b[1:] - a[1:] b[0] for the companion matrix A of a
    comp = np.zeros((n - 1, n - 1))
    comp[0, :] = -a[1:]
    for i in range(1, n - 1):
        comp[i, i - 1] = 1.0
    zi = np.linalg.solve(np.eye(n - 1) - comp.T, b[1:] - a[1:] * b[0])
    for v in (b, a, zi):
        v.setflags(write=False)
    return b, a, zi


class Event(Segment):
    """An event: a stretch of the file holding useful data (DataTypes.py:241-565)."""

    def __init__(self, current, segments=[], **kwargs):
        if len(segments):
            # an event given as its segments is the concatenation of their samples (nothing, if they have none)
            try:
                current = np.concatenate([piece.current for piece in segments])
            except Exception:
                current = ()
        super(Event, self).__init__(current, filtered=False, segments=segments, **kwargs)

    def filter(self, order=1, cutoff=2000.):
        """Zero-phase Bessel low-pass of ``self.current`` (DataTypes.py:258-274), on the device (csrc/filter.cuh)."""
        if type(self) is not Event:
            raise TypeError(_NEEDS_CURRENT)
        b, a, zi = bessel_coefficients(order, cutoff, self.second)
        samples = np.ascontiguousarray(self.current, dtype=np.float64)
        padlen = 3 * len(b)
        if samples.shape[0] <= padlen:
            raise ValueError("The length of the input vector x must be greater than padlen, which is %d." % padlen)
        ctx = _lib.default_context()
        ctx.upload_events_f64([samples])
        ctx.filter_events(b, a, zi)
        self.current = ctx.event_samples(samples.shape[0])
        self.filtered, self.filter_order, self.filter_cutoff = True, order, cutoff

    def parse(self, parser=SpeedyStatSplit(prior_segments_per_second=10), hmm=None):
        """Segment the event with a plug-in state parser (DataTypes.py:276-289,333); returns the segment count.

        With ``hmm`` (a ``pypore_b200.hmm.HMM``; the parser must be a ``SpeedyStatSplit``) the segment means are
        decoded with Viterbi and every run of consecutive segments in one state becomes one segment, whose
        statistics are computed again from the samples; each segment carries its ``state`` (-1 for every segment of
        an event whose sequence is impossible or holds a NaN)."""
        second = float(self.file.second)
        pieces = self._parse_hmm(parser, hmm) if hmm else parser.parse(self.current)
        for piece in pieces:
            piece.event = self
            piece.scale(second)
        self.segments, self.state_parser = pieces, parser
        return len(pieces)

    def _parse_hmm(self, parser, hmm):
        if not isinstance(parser, SpeedyStatSplit):
            raise TypeError("HMM-guided segmentation runs on the device with a SpeedyStatSplit parser")
        mw, MW, W, gain = parser._params()
        cur = SpeedyStatSplit._as_event(self.current)
        if cur.shape[0] == 0:
            return parser.parse(cur)
        ctx = _lib.default_context()
        ctx.upload_events_f64([cur])
        ctx.statsplit(mw, MW, W, gain)
        ctx.segment_stats()
        n = ctx.hmm_decode(hmm, "viterbi", merge=True)
        tab = ctx.segments(n)
        logp, states = ctx.hmm_download(1, n)
        self.log_probability = float(logp[0])
        pieces = []
        for k in range(n):
            a, b = int(tab["start"][k]), int(tab["end"][k])
            seg = Segment(current=cur[a:b], start=a, duration=b - a, end=b)
            seg._set_stats(tab["mean"][k], tab["std"][k], tab["min"][k], tab["max"][k])
            seg.state = int(states[k])
            pieces.append(seg)
        return pieces

    def apply_hmm(self, hmm, algorithm="viterbi"):
        """Decode the segment means with ``hmm`` (DataTypes.py:349-355): "viterbi" gives (log-probability, states),
        "forward" the log-likelihood."""
        means = np.array([seg.mean for seg in self.segments], dtype=np.float64)
        if algorithm == "viterbi":
            return hmm.viterbi(means)
        if algorithm == "forward":
            return hmm.log_probability(means)
        raise ValueError("algorithm must be 'viterbi' or 'forward', got %r" % (algorithm,))

    def delete(self):
        for name in ("current", "state_parser"):
            self.__dict__.pop(name, None)
        _each(self.segments, "delete")

    def to_meta(self):
        self._freeze(_STAT_SPAN, MetaEvent)
        _each(self.segments, "to_meta")

    def to_json(self, filename=None):
        return wire.dumps(wire.expand_event(self, strict=False), filename)

    @classmethod
    def from_json(cls, _json):
        """An Event if the JSON carries the samples, a MetaEvent otherwise (DataTypes.py:515-529)."""
        d = json.loads(wire.source_text(_json))
        if "current" in d:
            return cls(d["current"], start=d["start"])
        return MetaEvent(**d)

    n = property(lambda self: len(self.segments))


class _LazyList(object):
    """Sequence whose items are built on first access (object creation is the dominant host cost at 10^5..10^6
    segments, SURVEY 7.2 item 5).  ``untouched`` says that nothing has been handed out yet."""

    def __init__(self, n, factory):
        self._n, self._factory, self._cache = int(n), factory, {}

    untouched = property(lambda self: not self._cache)

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        item = self._cache.get(i)
        if item is None:
            item = self._cache[i] = self._factory(i)
        return item

    def __iter__(self):
        return (self[i] for i in range(self._n))

    def __add__(self, other):
        return list(self) + list(other)

    def __radd__(self, other):
        return list(other) + list(self)


class File(Segment):
    """A trace and the events detected in it (DataTypes.py:567-602).

    Only the ``current=`` / ``timestep=`` constructor is supported: there is no
    .abf data offline and the ABF reader is out of scope.  ``current`` may be an ``AdcTrace`` (int16 counts with
    their scale and offset): the parsers then work on the counts, and ``file.current`` is the decoded float64
    current, built on first access.
    """

    def __init__(self, filename=None, current=None, timestep=None, **kwargs):
        if current is None or timestep is None:
            if filename and current is None and timestep is None:
                raise NotImplementedError("reading .abf files is out of scope; pass current= and timestep=")
            raise SyntaxError("Must provide current and timestep, or filename corresponding to a valid abf file.")
        super(File, self).__init__(current=current, filename="", second=1000. / timestep, events=[], sample=None)
        if isinstance(current, AdcTrace):
            self.__dict__["_adc"] = self.__dict__.pop("current")

    def __getattr__(self, name):
        # only reached when `current` is not set: the AdcTrace's decoding, once
        adc = self.__dict__.get("_adc")
        if name != "current" or adc is None:
            raise AttributeError(name)
        current = self.__dict__["current"] = adc.decode()
        return current

    def __setattr__(self, name, value):
        if name == "current":
            self.__dict__.pop("_adc", None)   # other samples than the counts
        super(File, self).__setattr__(name, value)

    def _samples(self):
        """What the device parsers work on: the AdcTrace given as current=, else the current array."""
        adc = self.__dict__.get("_adc")
        return adc if adc is not None else np.asarray(self.current)

    __getitem__ = lambda self, index: self.events[index]     # noqa: E731
    n = property(lambda self: len(self.events))

    def parse(self, parser=lambda_event_parser(threshold=90), segmenter=None, filter_params=None,
              context=None, hmm=None):
        """Detect events with a plug-in event parser (DataTypes.py:589-602).

        With ``segmenter=`` (a ``SpeedyStatSplit``) the whole pipeline runs on the
        resident trace -- threshold scan, optional ``Event.filter(*filter_params)``,
        split search, statistics -- and every event comes back with its
        ``segments`` already parsed, as after ``event.parse(parser=segmenter)``.
        With ``hmm=`` (a ``pypore_b200.hmm.HMM``) one more device call decodes every event's segment means and
        merges runs of segments in one state, as after ``event.parse(parser=segmenter, hmm=hmm)``:
        ``segment_table`` gains a ``state`` column and ``event_table`` a ``log_probability`` column.
        """
        self.__dict__.pop("_tables", None)
        if hmm is not None and segmenter is None:
            raise ValueError("hmm= decodes segment means: it needs a segmenter")
        if segmenter is None and filter_params is None and not isinstance(parser, lambda_event_parser):
            # any duck-typed parser, exactly like the reference: seg.current / seg.start / seg.duration in samples
            rate, self.event_parser = self.second, parser
            self.events = [Event(current=seg.current, start=seg.start / rate,
                                 end=(seg.start + seg.duration) / rate, duration=seg.duration / rate,
                                 second=rate, file=self) for seg in parser.parse(self.current)]
            return
        if not isinstance(parser, lambda_event_parser):
            raise TypeError("the device-resident pipeline needs a pypore_b200 lambda_event_parser")
        self._parse_resident(context or _lib.default_context(), self._samples(), parser, segmenter, filter_params, hmm)

    # ------------------------------------------------------------------
    def _parse_resident(self, ctx, host, parser, segmenter, filter_params, hmm=None):
        filt = bessel_coefficients(filter_params[0], filter_params[1], self.second) if filter_params is not None else None
        rules = parser._device_rules()
        seg_table = None
        n_samples = host.shape[0]
        if segmenter is not None:
            mw, MW, W, gain = segmenter._params()
        if n_samples == 0:
            ev_start = ev_len = np.zeros(0, np.int64)
        elif rules is not None and segmenter is not None:
            # one call from host memory: the copy is chunked and overlapped with the stages (pp_pipeline_host)
            counts = _run_pipeline(ctx, host, parser.threshold, min_width=mw, max_width=MW, window_width=W,
                                   min_gain=gain, filter_ba=filt, with_stats=True, **rules.device_args())
            ev_start, ev_len = ctx.events(counts["events"])
            seg_table = ctx.segments(counts["segments"]) if hmm is None else None
        else:
            _upload_trace(ctx, host)
            ev_start, ev_len = parser._detect(ctx, host)[:2]
            if filt is not None and len(ev_start):
                ctx.filter_events(*filt)
            if segmenter is not None and len(ev_start):
                n_seg = ctx.statsplit(mw, MW, W, gain)
                ctx.segment_stats()
                seg_table = ctx.segments(n_seg) if hmm is None else None
        n_ev = len(ev_start)
        log_prob = None
        if hmm is not None:
            log_prob, state = np.zeros(0), np.zeros(0, np.int32)
            if n_ev:
                n_seg = ctx.hmm_decode(hmm, "viterbi", merge=True)
                seg_table = ctx.segments(n_seg)
                log_prob, state = ctx.hmm_download(n_ev, n_seg)
        ev_stats = ctx.event_stats(n_ev) if n_ev else {k: np.zeros(0) for k in ("mean", "std", "min", "max")}
        filtered = ctx.event_samples(int(ev_len.sum())) if filt is not None and n_ev else None
        if segmenter is not None and seg_table is None:
            seg_table = {"event": np.zeros(0, np.int32), "start": np.zeros(0, np.int64), "end": np.zeros(0, np.int64),
                         **{k: np.zeros(0) for k in ("mean", "std", "min", "max")}}
        self.event_table = dict(start=ev_start, length=ev_len, **ev_stats)
        if hmm is not None:
            seg_table["state"] = state
            self.event_table["log_probability"] = log_prob
        self.segment_table = seg_table
        self.event_parser = parser
        self._attach(wire.FileTables(self.second, self.event_table, seg_table, filter_params, segmenter),
                     host=host, filtered=filtered)

    def _attach(self, tables, host=None, filtered=None):
        """Make the file a view on `tables`: ``events`` builds Event / Segment objects (MetaEvent / MetaSegment for
        tables.meta) on demand."""
        self._tables = tables
        second = tables.second
        ev, sg = tables.events, tables.segments
        n_ev = len(ev["start"])
        ev_off = np.concatenate(([0], np.cumsum(ev["length"]))) if filtered is not None else None
        bounds = np.searchsorted(sg["event"], np.arange(n_ev + 1)) if sg is not None else None
        fp = tables.filter_params

        def span(a, n):
            return dict(start=a / second, end=(a + n) / second, duration=n / second)

        def stats(table, k):
            return table["mean"][k], table["std"][k], table["min"][k], table["max"][k]

        def meta_event(i):
            kw = dict(zip(("mean", "std", "min", "max"), stats(ev, i)))
            kw.update(span(int(ev["start"][i]), int(ev["length"][i])), second=second, file=self,
                      filtered=fp is not None, segments=[])
            if fp is not None:
                kw["filter_order"], kw["filter_cutoff"] = fp
            if sg is not None:
                lo = int(bounds[i])

                def meta_segment(j):
                    k = lo + j
                    a = int(sg["start"][k])
                    seg = MetaSegment(**dict(zip(("mean", "std", "min", "max"), stats(sg, k))),
                                      **span(a, int(sg["end"][k]) - a))
                    if "state" in sg:
                        seg.state = int(sg["state"][k])
                    return seg
                kw["segments"] = _LazyList(int(bounds[i + 1]) - lo, meta_segment)
                kw["state_parser"] = tables.state_parser
            return MetaEvent(**kw)

        def live_event(i):
            a, n = int(ev["start"][i]), int(ev["length"][i])
            samples = filtered[ev_off[i]:ev_off[i + 1]] if filtered is not None else np.array(host[a:a + n])
            event = Event(current=samples, second=second, file=self, **span(a, n))
            event._set_stats(*stats(ev, i))
            if "log_probability" in ev:
                event.log_probability = float(ev["log_probability"][i])
            if fp is not None:
                event.filtered, (event.filter_order, event.filter_cutoff) = True, fp
            if sg is not None:
                lo = int(bounds[i])

                def segment(j):
                    k = lo + j
                    s, e = int(sg["start"][k]), int(sg["end"][k])
                    seg = Segment(current=samples[s:e], start=s, duration=e - s, end=e)._set_stats(*stats(sg, k))
                    seg.event = event
                    if "state" in sg:
                        seg.state = int(sg["state"][k])
                    seg.scale(float(second))
                    return seg
                event.segments = _LazyList(int(bounds[i + 1]) - lo, segment)
                event.state_parser = tables.state_parser
            return event

        self.events = _LazyList(n_ev, meta_event if tables.meta else live_event)

    def _tables_current(self):
        """The tables still describe the file: no event object was handed out that the caller could have changed."""
        return isinstance(self.events, _LazyList) and self.events.untouched and "_tables" in self.__dict__

    def _segment_counts(self):
        """Segments per event, from the tables when they are current (no object is built for it)."""
        if self._tables_current():
            if self._tables.segments is None:
                return [0] * len(self.events)
            return np.bincount(np.asarray(self._tables.segments["event"], np.int64),
                               minlength=len(self.events)).tolist()
        return [event.n for event in self.events]

    def to_meta(self):
        """Drop the ionic current of the file and of everything under it (DataTypes.py:683-693)."""
        self.__dict__.pop("current", None)
        self.__dict__.pop("_adc", None)
        if self._tables_current():
            self._tables.meta = True
            self._attach(self._tables)
            return
        self.events = list(self.events)
        _each(self.events, "to_meta")

    def to_dict(self):
        """DataTypes.py:695-706 (a file with start and duration also gets its end)."""
        if not hasattr(self, "end") and hasattr(self, "start") and hasattr(self, "duration"):
            self.end = self.start + self.duration
        return wire.record(self, "File")

    def to_json(self, filename=None):
        """The file, its events and their segments as the reference's JSON (DataTypes.py:708-738)."""
        return wire.dumps(wire.file_tree(self), filename)

    @classmethod
    def from_json(cls, _json):
        """Rebuild a file from to_json's output (DataTypes.py:740-796).  The reference re-reads the .abf file named
        in the JSON and falls back to metadata objects when it cannot; reading .abf is out of scope here, so the
        result always holds MetaEvents / MetaSegments."""
        tree = json.loads(wire.source_text(_json))
        if tree["name"] != "File":
            raise TypeError("JSON does not encode a file")
        f = cls(current=[], timestep=1)
        f.event_parser = parser.from_json(json.dumps(tree["event_parser"]))
        f.events = []
        for row in tree["events"]:
            event = MetaEvent(**row)
            event.segments = [MetaSegment(**seg_row) for seg_row in row["segments"]]
            event.state_parser = parser.from_json(json.dumps(row["state_parser"]))
            event.filtered = row["filtered"]
            f.events.append(event)
        return f

    def delete(self):
        for name in ("current", "_adc", "event_parser", "_tables"):
            self.__dict__.pop(name, None)
        if isinstance(self.events, _LazyList):
            self.events = []
        _each(self.events, "delete")

    close = delete


class Experiment(object):
    """A series of files analysed together (DataTypes.py:938-1031).

    ``filenames`` may hold ``File`` objects (``File(current=..., timestep=...)``: the only way to get data in
    here, reading .abf is out of scope) next to file names; a name is handed to ``File(name)`` like the
    reference does.  ``parse`` keeps the reference's signature, defaults, printed messages and results; each
    file goes through ONE device-resident pass (threshold scan -> Event.filter -> segmenter -> statistics)
    instead of the reference's per-event Python loop.
    """

    def __init__(self, filenames, name=None):
        self.filenames, self.name, self.files = filenames, name or "Experiment", []

    @staticmethod
    def _report(file, with_segments):
        print("Opening {}".format(file.filename))
        print("\tDetected {} Events".format(file.n))
        if with_segments:
            for i, count in enumerate(file._segment_counts()):
                print("\t\tEvent {} has {} segments".format(i + 1, count))

    def parse(self, event_detector=lambda_event_parser(threshold=90),
              segmenter=SpeedyStatSplit(prior_segments_per_second=10, cutoff_freq=2000.),
              filter_params=(1, 2000), verbose=True, meta=False, batch=None):
        """DataTypes.py:956-988.  ``batch=`` (a ``pypore_b200.batch.FileBatch``; needs ``meta=True``, which
        discards the samples anyway) runs the files several at a time on the batch's worker contexts --
        and over its ranks, files being the unit -- and builds the same metadata objects from the gathered
        tables (kept as ``self.tables``)."""
        if batch is not None:
            return self._parse_batch(batch, event_detector, segmenter, filter_params, verbose, meta)
        on_device = (isinstance(event_detector, lambda_event_parser) and event_detector._device_rules() is not None
                     and (segmenter is None or isinstance(segmenter, SpeedyStatSplit))
                     and (segmenter is not None or filter_params is not None))
        for f in self._opened():
            if on_device:
                f.parse(parser=event_detector, segmenter=segmenter, filter_params=filter_params)
            else:
                # arbitrary Python rules or a foreign segmenter: per event, like the reference (DataTypes.py:972-982)
                f.parse(parser=event_detector)
                for ev in f.events:
                    if filter_params is not None:
                        ev.filter(*filter_params)
                    if segmenter is not None:
                        ev.parse(parser=segmenter)
            if verbose:
                self._report(f, segmenter is not None)
            if meta:
                f.to_meta()
            self.files += [f]

    def _opened(self):
        return (f if isinstance(f, File) else File(f) for f in self.filenames)

    def _parse_batch(self, batch, event_detector, segmenter, filter_params, verbose, meta):
        if not meta:
            raise ValueError("batch= keeps only the event / segment tables on the host; use it with meta=True")
        if segmenter is None:
            raise ValueError("batch= runs the whole pipeline; it needs a segmenter")
        if not (isinstance(event_detector, lambda_event_parser) and event_detector._device_rules() is not None
                and isinstance(segmenter, SpeedyStatSplit)):
            raise TypeError("batch= needs a lambda_event_parser with device-evaluable rules (parsers.RuleSet or the "
                            "defaults) and a SpeedyStatSplit; other plug-ins go through the sequential loop")
        files = list(self._opened())
        self.tables = batch.parse([f.current for f in files], [1000. / f.second for f in files], event_detector,
                                  segmenter, filter_params)
        for f in self.tables.files([f.filename for f in files], event_detector, segmenter, filter_params):
            if verbose:
                self._report(f, True)
            self.files += [f]

    def delete(self):
        _each(self.files, "delete")
        self.files = list()

    n = property(lambda self: len(self.files))

    @property
    def events(self):
        """All the events in all files."""
        return [event for file in self.files for event in file.events]

    @property
    def segments(self):
        """All segments of all events."""
        return [segment for event in self.events for segment in event.segments]


class Sample(object):
    """A container for events all suggested to be from the same substrate (DataTypes.py:1034-1040)."""

    def __init__(self, events=[], files=[], label=None):
        self.events, self.files, self.label = events, files, label

    def delete(self):
        _each(self.files, "delete")
