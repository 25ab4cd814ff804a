"""INTEGRATION.md section 1 for real: this repository's parsers handed to the REFERENCE's own containers.

The reference's plug-in boundary is duck-typed (`parser.parse(current) -> [Segment-like]`, PyPore/parsers.py:57-59):
`File.parse` reads `seg.current / seg.start / seg.duration` of what comes back (DataTypes.py:595-600), `Event.parse`
sets `segment.event` and calls `segment.scale(...)` (DataTypes.py:286-289), `File.to_json` asks the parsers for
`to_dict()` (DataTypes.py:729).  Here the reference's `File` / `Event` (loaded from /root/reference like the golden
fixtures were, tests/golden/make_golden.py) drive `pypore_b200.parsers.lambda_event_parser` and `SpeedyStatSplit`, and
the result is compared with the reference driving its OWN parsers on the same trace.

Those two tests need the reference's source tree: the CPU variant runs the plug-ins over an oracle-backed stand-in for
the device context (tests/oracle_device.py) and checks the protocol end to end; the `gpu` variant is the same test on
the real device.  Without the tree, the same run through this repository's own File / Event is still compared with
what the reference's File.to_json wrote for it (tests/golden/file_tierA.json, tests/golden/make_golden.py:golden_json)."""
import json
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from pypore_b200 import synth

REFERENCE = "/root/reference"
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, "PyPore")),
                                     reason="needs the original PyPore source tree, which is not part of this repository")


@pytest.fixture(scope="module")
def reference():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden
    return make_golden.load_reference()


def run(dt, P):
    """File.parse -> Event.filter on every other event -> Event.parse with File / Event from `dt` and the parsers of
    `P`: (the File, its to_json read back)."""
    x = synth.make_trace(4, seed=21, tier="A").astype(np.float64)
    rules = [lambda e: e.duration > 1000, lambda e: e.min > -0.5, lambda e: e.max < 110]
    kw = dict(min_width=100, window_width=10000, prior_segments_per_second=10, cutoff_freq=2000.)
    f = dt.File(current=x, timestep=0.01)
    f.parse(parser=P.lambda_event_parser(threshold=110, rules=rules))
    for i, event in enumerate(f.events):
        if i % 2 == 0:
            event.filter(1, 2000.)
        event.parse(parser=P.SpeedyStatSplit(**kw))
    return f, json.loads(f.to_json())


def run_both(reference):
    """(what the reference's File / Event produce with our plug-ins, what they produce with their own).  The filter
    is the reference's own scipy filter on both sides: the parsers see the same float64 samples."""
    from pypore_b200 import parsers as ours
    dt, ref_parsers, _ = reference
    return [run(dt, ours), run(dt, ref_parsers)]


def compare_json(j_ours, j_ref, stat_rtol):
    """Structure, parser state and every index equal; statistics to `stat_rtol`."""
    assert j_ours["n"] == j_ref["n"] == 4 and j_ours["event_parser"] == j_ref["event_parser"]
    for a, b in zip(j_ours["events"], j_ref["events"]):
        assert set(a) == set(b) and a["state_parser"] == b["state_parser"] and a["n"] == b["n"] > 1
        assert len(a["segments"]) == len(b["segments"]) == a["n"]
        for k in ("start", "end", "duration", "filtered", "name"):
            assert a[k] == b[k], k
        for sa, sb in zip(a["segments"], b["segments"]):
            assert (sa["start"], sa["end"], sa["duration"], sa["name"]) == (sb["start"], sb["end"], sb["duration"],
                                                                           sb["name"])
            for k in ("mean", "std", "min", "max"):
                assert abs(sa[k] - sb[k]) <= stat_rtol * abs(sb[k]), k


def check_segment_links(f_ours):
    """Our Segment objects inside the File's Event: scaled to seconds, linked to the event, sample views intact."""
    ev = f_ours.events[1]
    seg = ev.segments[1]
    assert seg.event is ev and abs(seg.duration * f_ours.second - len(seg.current)) < 1e-6
    assert np.array_equal(seg.current, ev.current[int(round(seg.start * f_ours.second)):][:len(seg.current)])


def compare(out, stat_rtol):
    (f_ours, j_ours), (f_ref, j_ref) = out
    assert type(f_ours.events[0]).__module__ == type(f_ref.events[0]).__module__     # the reference's Event class
    compare_json(j_ours, j_ref, stat_rtol)
    check_segment_links(f_ours)


def oracle_device(monkeypatch):
    from oracle_device import OracleDevice
    from pypore_b200 import _lib
    dev = OracleDevice()
    monkeypatch.setattr(_lib, "default_context", lambda device=None: dev)


def test_our_containers_and_parsers_match_the_references_json_oracle_device(monkeypatch):
    """This repository's File / Event and parsers over the oracle-backed device against the reference's stored
    File.to_json of the same run.  Event.filter is the oracle's restatement of scipy's filtfilt here (agrees with
    scipy to 1e-12 per sample, tests/test_oracle_golden.py)."""
    from pypore_b200 import DataTypes, parsers
    oracle_device(monkeypatch)
    f_ours, j_ours = run(DataTypes, parsers)
    j_ref = json.load(open(os.path.join(GOLDEN, "file_tierA.json")))
    compare_json(j_ours, j_ref, stat_rtol=1e-12)
    check_segment_links(f_ours)


@needs_reference
def test_reference_containers_drive_our_parsers_oracle_device(reference, monkeypatch):
    oracle_device(monkeypatch)
    compare(run_both(reference), stat_rtol=1e-12)


@needs_reference
@pytest.mark.gpu
def test_reference_containers_drive_our_parsers_on_the_device(reference):
    compare(run_both(reference), stat_rtol=1e-9)
