"""The sharded step's table path on ONE GPU: several contexts on device 0 play the ranks of tests/shard_cases.py and the
collectives become device copies (as in tests/test_gpu_dist.py::test_device_planned_step_on_one_gpu).  Per case:

- the device-planned step, and the host-planned redo (truncate, host plan, halo pieces appended from device or host
  memory, pp_shard_finish, the run-table rescan) whenever a rank raises flag 16 or 1;
- pp_pack_tables into the rows of one gathered buffer with sentinel padding, and once with a word too few;
- pp_unpack_tables into pinned host memory, into a device staging arena, on a caller stream, and for every contiguous
  range of ranks, against the per-rank downloads, the torch unpacking ShardedPipeline.tables uses and the oracle on the
  whole trace;
- two more steps on the same contexts (host-planned, then device-planned with another halo) giving the same tables;
- the refusals of pp_unpack_tables_range, and pp_pack_tables' refusal of tables whose extrema are not float32."""
import ctypes

import numpy as np
import pytest

import oracle
import shard_cases as shc

pytestmark = pytest.mark.gpu

SENTINEL = 0x5EC71E155EC71E15   # fits in int64: a word no packed or unpacked column holds here
COLS_I = ("ev_start", "ev_len", "seg_event", "seg_start", "seg_end")
COLS_F = ("mean", "std", "min", "max")


def _gain():
    from pypore_b200.parsers import statsplit_min_gain
    return statsplit_min_gain(**shc.SPLIT)


def _same_bits(a, b):
    """Bit for bit, except that any NaN equals any NaN (min / max pass through float32)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64))


def _assert_tables_equal(got, want, what, raw_bits=True):
    for k in COLS_I:
        assert np.array_equal(np.asarray(got[k], np.int64), want[k]), (what, k)
    for k in COLS_F:
        g, w = np.asarray(got[k], np.float64), want[k]
        if raw_bits and k in ("mean", "std"):
            assert np.array_equal(g.view(np.int64), w.view(np.int64)), (what, k)   # copied as raw 8-byte words
        else:
            assert _same_bits(g, w), (what, k)


def _oracle_tables(case):
    """The oracle on the whole trace, in the column layout of the unpacked tables."""
    x = case.x.astype(np.float64)
    ws, wl = oracle.events(x, shc.THRESHOLD, shc.rule_lambdas(case.rules))
    oe, ost, oen, _ = oracle.statsplit_events(x, ws, wl, gain=_gain()[3], threads=4)
    st = [[], [], [], []]
    for e in range(len(ws)):
        sel = oe == e
        a = int(ws[e])
        for j, v in enumerate(oracle.segment_stats(x[a:a + int(wl[e])], ost[sel], oen[sel])):
            st[j].append(v)
    st = [np.concatenate(v) if v else np.zeros(0) for v in st]
    return dict(ev_start=ws, ev_len=wl, seg_event=oe, seg_start=ost, seg_end=oen,
                mean=st[0], std=st[1], min=st[2], max=st[3])


def _assert_matches_oracle(t, o, what):
    for k in COLS_I:
        assert np.array_equal(t[k], o[k]), (what, k)
    for k in ("mean", "std"):
        assert np.allclose(t[k], o[k], rtol=1e-9, atol=0, equal_nan=True), (what, k)
    for k in ("min", "max"):
        assert _same_bits(t[k], o[k]), (what, k)


class Ranks(object):
    """One context per rank of `case`, every chunk resident with room for a halo behind it."""

    def __init__(self, case, f64=False):
        import torch
        from pypore_b200 import _lib
        self.case, self.world = case, case.world
        self.lens = case.lens()
        self.ctxs = []
        for r in range(self.world):
            c = _lib.Context(0)
            self.ctxs.append(c)
            if f64:
                c.upload_trace_f64(case.chunk(r))
            else:
                c.upload_trace(case.chunk(r), extra_capacity=shc.EXTRA_CAPACITY)
        self.recs = torch.zeros(self.world, 12, dtype=torch.float64, device="cuda")
        self.plans = torch.zeros(self.world, 8, dtype=torch.int64, device="cuda")
        self.res = torch.zeros(self.world, 8, dtype=torch.int64, device="cuda")
        self.mw, self.MW, self.W, self.gain = _gain()
        torch.cuda.synchronize()   # the contexts' streams do not wait for torch's

    def close(self):
        for c in self.ctxs:
            c.close()

    def sync(self):
        for c in self.ctxs:
            c.sync()

    def scan(self):
        for r, c in enumerate(self.ctxs):
            c.truncate_trace(self.lens[r])
            c.shard_scan(shc.THRESHOLD, self.lens[r], self.recs[r].data_ptr())
        self.sync()

    def device_step(self, halos):
        """scan -> stacked records -> the neighbour's head copied behind each chunk -> plan -> finish."""
        import torch
        from pypore_b200 import dist as ppdist
        rules = self.case.rules
        self.scan()
        dev = torch.device("cuda", 0)
        for r, c in enumerate(self.ctxs):
            if halos[r]:
                room = ppdist.device_view(c.trace_ptr + 4 * self.lens[r], halos[r], torch.float32, dev)
                room.copy_(ppdist.device_view(self.ctxs[r + 1].trace_ptr, halos[r], torch.float32, dev))
        torch.cuda.synchronize()
        for r, c in enumerate(self.ctxs):
            if halos[r]:               # pp_trace_extend takes float32 traces only, even for no samples
                c.extend_trace(halos[r])
            c.shard_plan(self.recs.data_ptr(), r, self.world, shc.THRESHOLD, rules, halos[r], self.plans[r].data_ptr())
            c.shard_finish_planned(shc.THRESHOLD, rules, self.mw, self.MW, self.W, self.gain, self.plans[r].data_ptr(),
                                   self.res[r].data_ptr())
        self.sync()
        return self.res.cpu().numpy()

    def host_step(self, from_host=False):
        """ShardedPipeline._step_host_planned: the run tables regrown and the chunks rescanned while any rank's
        overflowed, the host plan, the recv pieces appended, pp_shard_finish.  Returns (records, plans, rescans)."""
        import torch
        from pypore_b200 import dist as ppdist
        rules = self.case.rules
        rescans = 0
        for attempt in range(2):
            self.scan()
            infos = self.recs.cpu().numpy()
            if not infos[:, ppdist.I_PAD].any():
                break
            rescans += 1
            for r, c in enumerate(self.ctxs):
                c.threshold_scan(shc.THRESHOLD, scan_len=self.lens[r])
        else:
            raise AssertionError("run table overflow after the rescan")
        plans = ppdist.plan_boundaries(infos, rules)
        keep = []
        for r, c in enumerate(self.ctxs):
            for q, cnt in plans[r]["recv"]:
                if from_host:
                    piece = np.ascontiguousarray(self.case.chunk(q)[:cnt])
                    keep.append(piece)
                    c.append_trace(piece.ctypes.data, cnt, False)
                else:
                    c.append_trace(self.ctxs[q].trace_ptr, cnt, True)
            assert c.trace_len == self.lens[r] + shc.need(plans[r])
            p = plans[r]
            c.shard_finish(shc.THRESHOLD, rules, self.mw, self.MW, self.W, self.gain, p["skip_first"], p["skip_last"],
                           p["event"], self.res[r].data_ptr())
        self.sync()
        del keep
        return self.res.cpu().numpy(), plans, rescans

    def downloads(self, allr):
        """Commit every rank's record and download its tables: global event ids and starts, one array per column."""
        cols = {k: [] for k in COLS_I + COLS_F}
        base = 0
        for r, c in enumerate(self.ctxs):
            c.shard_commit(allr[r])
            ne, ns = int(allr[r, 1]), int(allr[r, 3])
            es, el = c.events(ne)
            sg = c.segments(ns)
            cols["ev_start"].append(es + self.case.cuts[r])
            cols["ev_len"].append(el)
            cols["seg_event"].append(sg["event"].astype(np.int64) + base)
            cols["seg_start"].append(sg["start"].copy())
            cols["seg_end"].append(sg["end"].copy())
            for k in COLS_F:
                cols[k].append(sg[k].copy())
            base += ne
        return {k: np.concatenate(v) if v else np.zeros(0) for k, v in cols.items()}


def _poison(views):
    """Overwrite a pinned arena's columns, so that a later unpack into it must really write every row."""
    for v in views.values():
        v.view(np.int64)[:] = SENTINEL


def _copy(views):
    return {k: np.array(v) for k, v in views.items()}


def _raw_unpack(c, g_ptr, world, m, allr_ptr, lo, hi, cap_e, cap_s, stream=None):
    """pp_unpack_tables_range into sentinel-filled device columns; returns (code, columns tensor [9, rows])."""
    import torch
    from pypore_b200 import _lib
    out = torch.full((9, max(cap_e, cap_s) + 8), SENTINEL, dtype=torch.int64, device="cuda")
    t = _lib.UnpackedTables()
    t.cap_events, t.cap_segments = int(cap_e), int(cap_s)
    for i, k in enumerate(COLS_I + COLS_F):
        setattr(t, k, out[i].data_ptr())
    torch.cuda.synchronize()
    code = c._L.pp_unpack_tables_range(c._h, ctypes.c_void_p(int(g_ptr)), int(world), int(m),
                                       ctypes.c_void_p(int(allr_ptr)), int(lo), int(hi), ctypes.byref(t), 0,
                                       ctypes.c_void_p(int(stream)) if stream else None)
    torch.cuda.synchronize()
    return code, out


def check_tables(ranks, allr, want_oracle, refusals=False):
    """Per-rank downloads against the oracle; packed, gathered and unpacked through every route against the downloads.
    Returns the downloaded columns."""
    import torch
    from pypore_b200 import _lib, dist as ppdist
    case, world = ranks.case, ranks.world
    dl = ranks.downloads(allr)
    _assert_matches_oracle(dl, want_oracle, case.name + ": per-rank downloads")
    counts = [(int(allr[r, 1]), int(allr[r, 3])) for r in range(world)]
    need = [2 * e + ppdist.SEG_WORDS * s for e, s in counts]
    m = (max(need) + 7) & ~1                                    # even, and longer than any rank needs
    sentinel = SENTINEL
    g = torch.full((world, m), sentinel, dtype=torch.int64, device="cuda")
    short = torch.full((world, m), sentinel, dtype=torch.int64, device="cuda")
    allr_dev = torch.from_numpy(np.ascontiguousarray(allr, np.int64)).cuda().view(-1)
    torch.cuda.synchronize()
    for r, c in enumerate(ranks.ctxs):
        c.pack_tables(allr_dev.data_ptr(), r, case.cuts[r], g[r].data_ptr(), m)
        if need[r]:
            c.pack_tables(allr_dev.data_ptr(), r, case.cuts[r], short[r].data_ptr(), need[r] - 1)
    ranks.sync()
    assert (short == sentinel).all(), (case.name, "packed with a word too few")
    for r in range(world):
        assert (g[r, need[r]:] == sentinel).all(), (case.name, r, "padding written")
        assert need[r] == 0 or (g[r, :need[r]] != sentinel).any(), (case.name, r, "nothing packed")
    E, S = sum(e for e, _ in counts), sum(s for _, s in counts)
    c0 = ranks.ctxs[0]

    # pinned host tables
    v = c0.unpack_tables(g.data_ptr(), world, m, allr_dev.data_ptr(), E, S)
    whole = _copy(v)
    _assert_tables_equal(whole, dl, case.name + ": pinned host")
    _poison(v)
    # device staging arena, then one copy to the host
    stage = torch.full((c0.unpacked_bytes(E, S),), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    v, arena = c0.unpack_tables(g.data_ptr(), world, m, allr_dev.data_ptr(), E, S, slot=1,
                                staging_ptr=stage.data_ptr())
    arena[:] = stage.cpu().numpy()
    _assert_tables_equal(_copy(v), dl, case.name + ": staging arena")
    _poison(v)
    # a caller stream: only enqueued there
    side = torch.cuda.Stream()
    v = c0.unpack_tables(g.data_ptr(), world, m, allr_dev.data_ptr(), E, S, stream=side.cuda_stream, slot=2)
    side.synchronize()
    _assert_tables_equal(_copy(v), dl, case.name + ": caller stream")
    _poison(v)
    # every contiguous range of ranks: the slice of the whole table
    eb = np.concatenate(([0], np.cumsum([e for e, _ in counts])))
    sb = np.concatenate(([0], np.cumsum([s for _, s in counts])))
    for lo in range(world):
        for hi in range(lo + 1, world + 1):
            ne, ns = int(eb[hi] - eb[lo]), int(sb[hi] - sb[lo])
            v = c0.unpack_tables(g.data_ptr(), world, m, allr_dev.data_ptr(), ne, ns, slot=3, ranks=(lo, hi))
            part = {k: (whole[k][eb[lo]:eb[hi]] if k.startswith("ev_") else whole[k][sb[lo]:sb[hi]]) for k in whole}
            _assert_tables_equal(_copy(v), part, "%s: ranks %d..%d" % (case.name, lo, hi))
            _poison(v)
    # the torch path of ShardedPipeline.tables
    t = ppdist.unpack_gathered(g, counts)
    _assert_tables_equal(ppdist.columns({k: u.cpu().numpy() for k, u in t.items()}), dl, case.name + ": torch")

    if refusals:
        def untouched(code, out, want, what):
            assert code == want, (case.name, what, code)
            assert (out == sentinel).all(), (case.name, what, "output written")
        if E:
            untouched(*_raw_unpack(c0, g.data_ptr(), world, m, allr_dev.data_ptr(), 0, world, E - 1, S),
                      _lib.PP_ERR_CAPACITY, "cap_events")
        if S:
            untouched(*_raw_unpack(c0, g.data_ptr(), world, m, allr_dev.data_ptr(), 0, world, E, S - 1),
                      _lib.PP_ERR_CAPACITY, "cap_segments")
        untouched(*_raw_unpack(c0, g.data_ptr(), world, m - 1, allr_dev.data_ptr(), 0, world, E, S),
                  _lib.PP_ERR_ARG, "odd words_per_rank")
        big = torch.zeros(65 * 8, dtype=torch.int64, device="cuda")
        untouched(*_raw_unpack(c0, g.data_ptr(), 65, m, big.data_ptr(), 0, 65, E, S), _lib.PP_ERR_ARG, "world 65")
        lo = 1 if world > 1 else 0
        untouched(*_raw_unpack(c0, g.data_ptr(), world, m, allr_dev.data_ptr(), lo, lo, E, S), _lib.PP_ERR_ARG,
                  "empty rank range")
        # words_per_rank two words short of the longest rank: the rows of every rank, cut to that length as an
        # all-gather of the first m words would, at that stride.  Rank rows past the cut would be read from the next
        # rank's row (or the slack behind the last), never further, so even a kernel without the check stays inside.
        ms = max(need) - 2
        gs = torch.full((world * ms + 64,), sentinel, dtype=torch.int64, device="cuda")
        for r in range(world):
            gs[r * ms:(r + 1) * ms] = g[r, :ms]
        untouched(*_raw_unpack(c0, gs.data_ptr(), world, ms, allr_dev.data_ptr(), 0, world, E, S),
                  _lib.PP_ERR_CAPACITY, "words_per_rank short")
        untouched(*_raw_unpack(c0, gs.data_ptr(), world, ms, allr_dev.data_ptr(), 0, world, E, S,
                               stream=side.cuda_stream), _lib.PP_OK, "words_per_rank short, caller stream")
        # the same call with enough words per rank unpacks (the refusals above are about the arguments only)
        code, out = _raw_unpack(c0, g.data_ptr(), world, m, allr_dev.data_ptr(), 0, world, E, S)
        assert code == _lib.PP_OK
        o = out.cpu().numpy()
        got = {k: o[i, :E if k.startswith("ev_") else S] for i, k in enumerate(COLS_I)}
        got.update({k: o[5 + i, :S].view(np.float64) for i, k in enumerate(COLS_F)})
        _assert_tables_equal(got, dl, case.name + ": device columns")
    return dl


def _flags(allr):
    return int(np.bitwise_or.reduce(allr[:, 4] & 17))


@pytest.mark.parametrize("name", sorted(shc.cases()))
def test_sharded_tables_match_downloads_and_oracle(name):
    case = shc.cases()[name]
    t = case.targets
    want = _oracle_tables(case)
    ranks = Ranks(case)
    try:
        # step 1: device-planned, redone with the host plan when a rank asks for it
        allr = ranks.device_step(case.halos())
        assert _flags(allr) == t["redo"]
        if t["redo"]:
            allr, plans, rescans = ranks.host_step(from_host=case.host_halo)
            assert _flags(allr) == 0 and rescans == (1 if t["overflow"] else 0)
            for r in t["span3"]:
                assert len(plans[r]["recv"]) >= 2 and ranks.ctxs[r].trace_len >= ranks.lens[r] + ranks.lens[r + 1]
        for r in t["empty"]:
            assert allr[r, 1] == 0 and allr[r, 3] == 0
        assert all(allr[r, 1] > 0 for r in range(case.world) if r not in t["empty"])
        first = check_tables(ranks, allr, want, refusals=True)
        # step 2: host-planned on the same contexts
        allr, plans, _ = ranks.host_step()
        assert _flags(allr) == 0
        _assert_tables_equal(check_tables(ranks, allr, want), first, case.name + ": host-planned step")
        # step 3: device-planned after it, the halo now exactly what each single-piece owner needs
        halos = [shc.need(p) if len(p["recv"]) == 1 else h for p, h in zip(plans, case.halos())]
        allr = ranks.device_step(halos)
        assert _flags(allr) & ~16 == 0 and bool(_flags(allr)) == bool(t["span3"])
        if _flags(allr):
            allr, _, rescans = ranks.host_step()
            assert rescans == 0          # the run tables kept the capacity the rescan gave them
        _assert_tables_equal(check_tables(ranks, allr, want), first, case.name + ": device-planned after host-planned")
    finally:
        ranks.close()


def _pack_code(c, allr_row, m=4096):
    """pp_pack_tables of `c`'s tables as rank 0 of one; returns (code, output untouched)."""
    import torch
    sentinel = SENTINEL
    rec = torch.from_numpy(np.ascontiguousarray(allr_row, np.int64)).cuda()
    out = torch.full((m,), sentinel, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    code = c._L.pp_pack_tables(c._h, ctypes.c_void_p(rec.data_ptr()), 0, 0, ctypes.c_void_p(out.data_ptr()), m)
    c.sync()
    return code, bool((out == sentinel).all()), out


def test_float64_ranks_work_and_their_tables_are_not_packed():
    """Float64 ranks scan, plan and finish with exact tables, but their extrema are not float32 values: packing them
    is refused, as after a pipeline on an ADC trace, on filtered events or on uploaded float64 events."""
    from pypore_b200 import _lib, dist as ppdist
    from pypore_b200.adc import AdcTrace
    from pypore_b200.DataTypes import bessel_coefficients
    x, cuts = shc.f64_trace()
    case = shc.Case("f64", x, cuts, halo=0)
    want = _oracle_tables(case)
    ranks = Ranks(case, f64=True)
    try:
        allr = ranks.device_step(case.halos())
        assert _flags(allr) == 0
        plans = ppdist.plan_boundaries(ranks.recs.cpu().numpy(), case.rules)
        assert plans[0]["skip_last"] and plans[0]["event"] is None        # the cut is in the open channel
        dl = ranks.downloads(allr)
        _assert_matches_oracle(dl, want, "float64 ranks")
        assert (dl["min"].astype(np.float32).astype(np.float64) != dl["min"]).any()
        for r, c in enumerate(ranks.ctxs):
            code, untouched, _ = _pack_code(c, allr[r])
            assert code == _lib.PP_ERR_STATE and untouched, r
    finally:
        ranks.close()

    x32 = shc.synth.make_trace(4, seed=76)
    mw, MW, W, gain = _gain()
    rules = shc.RULES7
    args = (shc.THRESHOLD, rules["rule_mask"], rules["duration_gt"], rules["duration_lt"], rules["min_gt"],
            rules["max_lt"], mw, MW, W, gain)
    c = _lib.Context(0)
    try:
        def record(res):
            return [res["runs"], res["events"], res["event_samples"], res["segments"], 0, 0, 0, 0]
        # float32 trace: packed, and min / max come back exactly
        c.upload_trace(x32)
        res = c.pipeline(*args)
        code, _, out = _pack_code(c, record(res))
        assert code == _lib.PP_OK
        sg = c.segments(res["segments"])
        w = out.cpu().numpy()[2 * res["events"]:2 * res["events"] + 4 * res["segments"]].reshape(-1, 4)
        mnmx = w[:, 3].copy().view(np.float32).reshape(-1, 2).astype(np.float64)
        assert _same_bits(mnmx[:, 0], sg["min"]) and _same_bits(mnmx[:, 1], sg["max"])
        # the same trace filtered: the events' samples are float64
        res = c.pipeline(*args, filter_ba=bessel_coefficients(1, 2000., 1e5))
        assert res["segments"] > 0 and _pack_code(c, record(res))[:2] == (_lib.PP_ERR_STATE, True)
        # ADC counts at a scale float32 cannot hold
        counts = np.round(x32.astype(np.float64) * 32).astype(np.int16)
        c.upload_trace_adc16(AdcTrace(counts, 0.0305, 0.0123))
        res = c.pipeline(*args)
        assert res["segments"] > 0 and _pack_code(c, record(res))[:2] == (_lib.PP_ERR_STATE, True)
        # uploaded float64 events
        arrays = [x32[:7000].astype(np.float64) * 0.0305 * 32 + 0.0123, np.linspace(20.0, 21.0, 3000) + 1e-9]
        lens = c.upload_events_f64(arrays)
        ns = c.statsplit(mw, MW, W, gain)
        c.segment_stats()
        rec = [0, len(lens), int(lens.sum()), ns, 0, 0, 0, 0]
        assert ns > 0 and _pack_code(c, rec)[:2] == (_lib.PP_ERR_STATE, True)
    finally:
        c.close()
