"""The cases of tests/test_gpu_shard_tables.py reach what they were built for (no GPU): which boundaries join, which
straddling events the speculative halo covers, which joined runs the rules reject, the event over three chunks, the
ranks without events, the run-table overflow and the redo flags the device plan raises.  Every rank's boundary record
is built from the oracle's runs of its chunk and planned with pypore_b200.dist.plan_boundaries, as the host-planned
step does."""
import numpy as np
import pytest

import oracle
import shard_cases as shc
from pypore_b200 import dist as ppdist


def device_redo(case, infos, plans, halos):
    """The redo flags k_shard_plan raises (threshold.cuh): 16 when an accepted straddling event needs more than the
    speculative halo or more than one neighbour, 1 when any rank's run table overflowed."""
    flags = 0
    for r, p in enumerate(plans):
        if p["event"] is not None and (len(p["recv"]) > 1 or shc.need(p) > halos[r]):
            flags |= 16
    for r in range(case.world):
        if len(shc.runs(case.chunk(r))[0]) > case.lens()[r] // 256 + 4096:
            flags |= 1
    return flags


def sharded_events(case, plans):
    """Global (start, length) of the events the ranks select under the plan: the chunk's own runs minus the ones a
    neighbour decides, plus the straddling event the rank owns."""
    starts, lens = [], []
    for r, p in enumerate(plans):
        c = case.chunk(r).astype(np.float64)
        runs = list(shc.runs(c))
        keep = set(oracle.select_runs(c, runs, shc.rule_lambdas(case.rules)).tolist())
        if p["skip_first"]:
            keep.discard(0)
        if p["skip_last"]:
            keep.discard(len(runs[0]) - 1)
        for i in sorted(keep):
            starts.append(case.cuts[r] + int(runs[0][i]))
            lens.append(int(runs[1][i]))
        if p["event"] is not None:
            starts.append(case.cuts[r] + p["event"][0])
            lens.append(p["event"][1])
    return np.asarray(starts, np.int64), np.asarray(lens, np.int64)


@pytest.mark.parametrize("name", sorted(shc.cases()))
def test_case_reaches_its_plan_shape(name):
    case = shc.cases()[name]
    t = case.targets
    infos = shc.infos(case)
    plans = shc.plans(case)
    halos = case.halos()
    world = case.world
    assert case.cuts[0] == 0 and case.cuts[-1] == case.n and all(l > 0 for l in case.lens())
    joins = [bool(infos[b][ppdist.I_LAST_BELOW] == infos[b + 1][ppdist.I_FIRST_BELOW]) for b in range(world - 1)]
    assert [b for b in range(world - 1) if joins[b]] == list(t["joined"])
    for b in range(world - 1):
        owns = joins[b] and not (infos[b][ppdist.I_NRUNS] == 1 and plans[b]["skip_first"])
        p = plans[b]
        if b in t["covered"]:
            assert p["event"] is not None and len(p["recv"]) == 1 and shc.need(p) <= halos[b]
        if b in t["rejected"]:
            assert owns and p["skip_last"] and p["event"] is None and p["recv"] == []
        elif owns:
            assert p["event"] is not None
    for r in t["span3"]:
        assert plans[r]["event"] is not None and len(plans[r]["recv"]) >= 2
    accepted = [r for r in range(world) if plans[r]["event"] is not None]
    assert [r for r in accepted if len(plans[r]["recv"]) == 1 and shc.need(plans[r]) <= halos[r]] == list(t["covered"])
    assert all(shc.need(plans[r]) <= shc.EXTRA_CAPACITY for r in accepted)
    ws, wl = shc.events_of(case.x, case.rules)
    owner = np.searchsorted(np.asarray(case.cuts), ws, side="right") - 1
    assert [r for r in range(world) if not (owner == r).any()] == list(t["empty"])
    assert device_redo(case, infos, plans, halos) == t["redo"]
    assert [r for r in range(world) if len(shc.runs(case.chunk(r))[0]) > case.lens()[r] // 256 + 4096] == \
        list(t["overflow"])
    # the plan loses and duplicates nothing: the ranks' events are the oracle's events of the whole trace
    ss, sl = sharded_events(case, plans)
    order = np.argsort(ss, kind="stable")
    assert np.array_equal(ss[order], ws) and np.array_equal(sl[order], wl)


def test_world_sizes_and_every_target_are_present():
    cs = shc.cases().values()
    assert {c.world for c in cs} == {1, 2, 3, 5}
    for key in ("covered", "rejected", "span3", "empty", "overflow"):
        assert any(c.targets[key] for c in cs), key
    assert {c.targets["redo"] for c in cs} == {0, 1, 16}
    assert any(c.host_halo for c in cs)


def test_cuts_sit_where_the_cases_say():
    cs = shc.cases()
    c = cs["w3_event_edges"]
    ws, wl = shc.events_of(c.x)
    assert c.cuts[1] in set(ws.tolist()) and c.cuts[2] in set((ws + wl).tolist())
    p = shc.plans(c)
    assert all(not q["skip_first"] and not q["skip_last"] for q in p)
    # the halo exactly at the owner's need, and one sample short of it
    for name, short in (("w2_halo_at_need", 0), ("w2_halo_short", 1)):
        c = cs[name]
        assert c.halos()[0] == shc.need(shc.plans(c)[0]) - short
    c = cs["w2_nan_edge"]
    x = c.x
    assert np.isnan(x[c.cuts[1]]) and x[c.cuts[1] - 1] < 110 and x[c.cuts[1] + 1] < 110
    # the three-chunk event: all of rank 2's chunk and the head of rank 3's
    c = cs["w5_span3"]
    p = shc.plans(c)
    assert [q for q, _ in p[1]["recv"]] == [2, 3] and p[1]["recv"][0][1] == c.lens()[2]
    assert p[2]["skip_first"] and p[2]["skip_last"] and p[2]["event"] is None


def test_rejected_straddlers_fail_only_once_joined():
    c = shc.cases()["w3_rejected"]
    infos = shc.infos(c)
    rules = c.rules
    # the short event: each part and the joined run are short
    joined = infos[0][ppdist.I_LAST_LEN] + infos[1][ppdist.I_FIRST_LEN]
    assert joined <= rules["duration_gt"] and joined == 800
    # the spike: the left part alone passes every rule, the joined run fails MIN_GT only
    left = (infos[1][ppdist.I_LAST_LEN], infos[1][ppdist.I_LAST_MIN], infos[1][ppdist.I_LAST_MAX])
    assert ppdist.rules_accept(rules, *left)
    mn = min(infos[1][ppdist.I_LAST_MIN], infos[2][ppdist.I_FIRST_MIN])
    mx = max(infos[1][ppdist.I_LAST_MAX], infos[2][ppdist.I_FIRST_MAX])
    assert mn < rules["min_gt"] and ppdist.rules_accept(dict(rules, rule_mask=5),
                                                        left[0] + infos[2][ppdist.I_FIRST_LEN], mn, mx)


def test_non_finite_case_has_minus_inf_and_minus_zero_segments():
    c = shc.cases()["w3_non_finite"]
    x = c.x.astype(np.float64)
    ws, wl = shc.events_of(c.x, c.rules)
    from pypore_b200.parsers import statsplit_min_gain
    gain = statsplit_min_gain(**shc.SPLIT)[3]
    oe, ost, oen, _ = oracle.statsplit_events(x, ws, wl, gain=gain, threads=4)
    mean, std, mn, mx = [], [], [], []
    for e in range(len(ws)):
        sel = oe == e
        a = int(ws[e])
        m, s, lo, hi = oracle.segment_stats(x[a:a + wl[e]], ost[sel], oen[sel])
        mean.append(m), std.append(s), mn.append(lo), mx.append(hi)
    mean, std, mn = np.concatenate(mean), np.concatenate(std), np.concatenate(mn)
    inf = np.isneginf(mn)
    assert inf.any() and np.isneginf(mean[inf]).all() and np.isnan(std[inf]).all()
    zero = (mn == 0) & np.signbit(mn)
    assert zero.any()
    # the -inf sample is in the right-hand part of the straddling event, which rank 0 owns
    b = c.cuts[1]
    assert np.isneginf(x[b:]).any() and not np.isneginf(x[:b]).any()
    assert np.isneginf(x[b:c.cuts[1] + shc.need(shc.plans(c)[0])]).any()
