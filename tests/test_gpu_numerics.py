"""The numeric kernels around the split search, each against an exact or bit-exact reference of the same
operation, on every sample source (float32 trace, float64 trace, int16 ADC trace, packed float64 events):

* K2 prefix sums: bit for bit np.cumsum(x) / np.cumsum(x * x), and the exactness verdict against a restatement
  of the proof (prefix.cuh) from the samples' bit patterns;
* K4 statistics: mean / std against the exact values (integer arithmetic, rounded once), min / max bitwise;
* K5 filter: orders 3-8 bit for bit the oracle's sequential filtfilt with the same b, a, zi; orders 1-2 (the
  parallel scan) within 1e-8 of the largest |y| of the event.

Rows are placed at every 16-byte phase of the trace (start offsets 0-7 samples), the samples between them are
NaN (ADC: the int16 extremes), so a kernel that reads outside a row shows.  Measured worst errors are printed
(run with -s to see them).
"""
import ctypes
import math
from fractions import Fraction

import numpy as np
import pytest

import oracle
from oracle import oracle as orc
from pypore_b200 import _lib
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import bessel_coefficients

pytestmark = pytest.mark.gpu

STAT_RTOL = 1e-9


class Content(object):
    """The same float64 rows for every source kind: decoded samples, given either directly or as int16 counts
    with the decoding counts * scale + offset."""

    def __init__(self, rows=None, counts=None, scale=None, offset=0.0):
        if counts is not None:
            self.counts = [np.ascontiguousarray(c, np.int16) for c in counts]
            self.scale, self.offset = float(scale), float(offset)
            self.rows = [c.astype(np.float64) * self.scale + self.offset for c in self.counts]
        else:
            self.counts = None
            self.rows = [np.ascontiguousarray(r, np.float64) for r in rows]

        self.verdicts = {}   # float32 rule? -> restated exactness verdict per row

    def kinds(self):
        """The source kinds that hold this content exactly."""
        with np.errstate(over="ignore"):
            f32 = all(np.array_equal(r.astype(np.float32).astype(np.float64), r, equal_nan=True) for r in self.rows)
        return (["trace32"] if f32 else []) + ["trace64"] + (["adc16"] if self.counts is not None else []) + \
            ["flat64"]

    def lengths(self):
        return np.array([len(r) for r in self.rows], np.int64)


def put(ctx, kind, content, phase=0):
    """Make `content` resident as the rows (events) of `kind`.  On a trace, row i starts at a sample offset
    congruent to i + phase modulo 8, behind at least one padding sample."""
    if kind == "flat64":
        ctx.upload_events_f64(content.rows)
        return
    starts, pos = [], 0
    for i, r in enumerate(content.rows):
        s = pos + 1
        s += (i + phase - s) % 8
        starts.append(s)
        pos = s + len(r)
    n = pos + 9
    if kind == "adc16":
        buf = np.full(n, 32767, np.int16)
        buf[::2] = -32768
        for s, c in zip(starts, content.counts):
            buf[s:s + len(c)] = c
        ctx.upload_trace_adc16(AdcTrace(buf, content.scale, content.offset))
    else:
        buf = np.full(n, np.nan, np.float32 if kind == "trace32" else np.float64)
        for s, r in zip(starts, content.rows):
            buf[s:s + len(r)] = r
        if kind == "trace32":
            ctx.upload_trace(buf)
        else:
            ctx.upload_trace_f64(buf)
    ctx.set_events(starts, content.lengths())


def same_bits(a, b):
    """Bitwise equal, NaN positions equal (the payload of a NaN is not compared)."""
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


# ------------------------------------------------------------------------------------------- K2 prefix sums
def exponents(v, f32):
    """Per sample: (lowest set bit exponent, magnitude exponent, finite and non-zero) from the bit pattern of
    v as float32 (f32) or float64.  Denormals: the magnitude exponent of the smallest normal minus one for
    float64 (|v| < 2^-1022), and for float32 -126 (|v| < 2^-125) -- what the device takes per path is below."""
    if f32:
        b = v.astype(np.float32).view(np.uint32).astype(np.int64)
        E, m, mbits, bias = (b >> 23) & 0xff, b & 0x7fffff, 23, 127
        special = E == 0xff
    else:
        b = v.view(np.uint64)
        E = ((b >> np.uint64(52)) & np.uint64(0x7ff)).astype(np.int64)
        m = (b & np.uint64(0xfffffffffffff)).astype(np.int64)
        mbits, bias = 52, 1023
        special = E == 0x7ff
    sig = np.where(E > 0, m | (1 << mbits), m)
    nz = sig != 0
    s = np.where(nz, sig, 1)
    ctz = np.log2(s & -s).astype(np.int64)       # s & -s: the lowest set bit, an exact power of two
    elow = np.maximum(E, 1) - bias - mbits + ctz
    emax = np.where(E > 0, E - bias, -bias if not f32 else -126)
    return elow, emax, nz & ~special, special


def restated_verdict(x, f32, long_path):
    """prefix.cuh's exactness test for one event: ceil(log2 n) + emax + 1 - elow <= 53, for x and for fl(x*x)
    (float32 samples: x*x is exact, its exponents are 2 elow and 2 emax + 1).  inf / NaN: never exact."""
    n = len(x)
    lg = int(math.ceil(math.log2(n))) if n > 1 else 0

    def ok(v, vf32, sq):
        el, em, live, special = exponents(v, vf32)
        if special.any():
            return False
        if not live.any():
            return True
        lo, hi = int(el[live].min()), int(em[live].max())
        if vf32 and long_path and hi == -126 and not (v.astype(np.float32).view(np.uint32) & 0x7f800000).any():
            hi = -127          # the tiled kernels' float32 exponents take a denormal maximum as 2^-127
        if sq:
            lo, hi = 2 * lo, 2 * hi + 1
        return lg + hi + 1 - lo <= 53

    if f32:
        return ok(x, True, False) and ok(x, True, True)
    with np.errstate(over="ignore", under="ignore", invalid="ignore"):
        return ok(x, False, False) and ok(x * x, False, False)


def prefix_families():
    rng = np.random.RandomState(20)
    lengths = [1, 2, 255, 256, 257, 2047, 2048, 2049, 32767, 32768, 32769, 100003, 3000017]

    def counts(n):
        return np.clip(rng.normal(0, 4000, n), -32000, 32000).astype(np.int16)

    fams = {   # dyadic: |x| < 2^9 in steps of 2^-6, proven exact up to 2^22 samples even by the float32 rule
        "adc_dyadic": Content(counts=[counts(n) for n in lengths], scale=2.0 ** -6, offset=0.25),
        "adc_nondyadic": Content(counts=[counts(n) for n in lengths], scale=0.0305, offset=0.0123),
        "adc_negative": Content(counts=[counts(n) for n in lengths], scale=-0.0625, offset=3.5),
        "raw_float32": Content(rows=[rng.normal(60, 2, n).astype(np.float32) for n in lengths]),
    }
    tiny = 2.0 ** -149

    def noise(n):
        return rng.normal(0, 1, n).astype(np.float32)

    fams["special32"] = Content(rows=[   # float32-exact: on every float kind
        np.zeros(300), np.zeros(40000),
        rng.randint(-1000, 1000, 3000) * tiny,                                   # float32 denormals
        np.r_[1.5, rng.randint(1, 9, 40000) * tiny],                             # ... beside a normal sample
        np.r_[noise(100), np.inf, noise(100)], np.r_[-np.inf, noise(40000)], np.r_[noise(5000), np.nan],
        np.r_[np.full(3, np.inf), np.full(3, -np.inf)]])
    fams["denormal64"] = Content(rows=[rng.randint(-7, 8, 3000) * 5e-324, rng.randint(-7, 8, 40000) * 5e-324,
                                       np.r_[1.0, rng.randint(-7, 8, 300) * 5e-324]])
    return fams


@pytest.fixture(scope="module")
def prefix_data():
    fams = prefix_families()
    refs = {}
    for name, c in fams.items():
        with np.errstate(over="ignore", invalid="ignore"):
            refs[name] = [(np.cumsum(r), np.cumsum(r * r)) for r in c.rows]
    return fams, refs


def check_prefix(ctx, kind, content, refs, mode):
    """One pp_prefix run: every event bitwise np.cumsum (PARALLEL: only those the proof covers), the redo flags
    event by event the restated verdict.  Returns the number of events the proof covers."""
    put(ctx, kind, content)
    ctx.prefix(mode)
    lens = content.lengths()
    c, c2, redone = ctx.debug_prefix(len(lens), int(lens.sum()))
    off = np.r_[0, np.cumsum(lens)]
    f32 = kind == "trace32"
    if f32 not in content.verdicts:
        content.verdicts[f32] = np.array([restated_verdict(r, f32, len(r) > 32768) for r in content.rows])
    exact = content.verdicts[f32]
    if mode == _lib.PREFIX_AUTO:
        assert np.array_equal(redone, ~exact), (kind, np.nonzero(redone != ~exact)[0], lens[redone != ~exact])
    else:
        assert redone.all() if mode == _lib.PREFIX_SEQUENTIAL else not redone.any()
    for e, (rc, rc2) in enumerate(refs):
        if mode == _lib.PREFIX_PARALLEL and not exact[e]:
            continue
        assert same_bits(c[off[e]:off[e + 1]], rc), (kind, mode, e, lens[e], "c")
        assert same_bits(c2[off[e]:off[e + 1]], rc2), (kind, mode, e, lens[e], "c2")
    return int(exact.sum())


@pytest.mark.parametrize("family", ["adc_dyadic", "adc_nondyadic", "adc_negative", "raw_float32", "special32",
                                    "denormal64"])
def test_prefix_bitwise_every_source_and_mode(ctx, prefix_data, family):
    """K2 against np.cumsum bit for bit: short events (one warp, <= 32768 samples), the tiled reduce / carries /
    scan above that, one event of 3 M samples; AUTO and SEQUENTIAL everywhere, PARALLEL where the proof holds."""
    fams, refs = prefix_data
    content = fams[family]
    for kind in content.kinds():
        for mode in (_lib.PREFIX_AUTO, _lib.PREFIX_SEQUENTIAL, _lib.PREFIX_PARALLEL):
            proven = check_prefix(ctx, kind, content, refs[family], mode)
        if family == "adc_dyadic":
            assert proven == len(content.rows)      # quantised data is proven exact: no redo
        if family in ("adc_nondyadic", "raw_float32"):
            assert proven < len(content.rows)


def test_prefix_verdict_at_the_53_bit_boundary(ctx):
    """Multiples of 1/32 below 2^14 (ADC: counts / 32 + 15360): fl(x*x) < 2^28 in steps of 2^-10, so
    ceil(log2 n) + 27 + 1 + 10 is 53 at n = 32768 (proven) and 54 at n = 32769 (across the short / tiled path
    switch) and n = 65536.  The flags equal the restatement on every source kind, AUTO equals np.cumsum, and the
    54-bit event really rounds: PARALLEL differs from np.cumsum there."""
    rng = np.random.RandomState(21)
    lens = (32768, 32769, 65536)
    cnt = [rng.randint(-32768, 32768, n).astype(np.int16) for n in lens]
    for c in cnt:
        c[0], c[1] = 32767, -32767              # the largest |x| (just below 2^14) and an odd count
    content = Content(counts=cnt, scale=2.0 ** -5, offset=15360.0)
    refs = [(np.cumsum(r), np.cumsum(r * r)) for r in content.rows]
    assert [restated_verdict(r, False, n > 32768) for r, n in zip(content.rows, lens)] == [True, False, False]
    kinds = content.kinds()
    assert kinds == ["trace32", "trace64", "adc16", "flat64"]
    for kind in kinds:
        assert check_prefix(ctx, kind, content, refs, _lib.PREFIX_AUTO) == 1
        put(ctx, kind, content)
        ctx.prefix(_lib.PREFIX_PARALLEL)
        c, c2, _ = ctx.debug_prefix(3, sum(lens))
        assert c2[:32768].tobytes() == refs[0][1].tobytes()
        assert c2[32768 + 32769:].tobytes() != refs[2][1].tobytes(), kind


# ------------------------------------------------------------------------------------------- K4 statistics
def exact_stats(x):
    """Exact mean and variance of finite float64 samples (integers scaled to a common exponent), each rounded
    once to float64; std = sqrt of the rounded variance."""
    m, e = np.frexp(x)
    mi = np.ldexp(m, 53).astype(np.int64).astype(object)
    ei = e.astype(np.int64) - 53
    e0 = int(ei.min())
    v = mi * np.array([1 << int(k) for k in (ei - e0)], dtype=object)
    n = len(x)
    s1, s2 = int(v.sum()), int((v * v).sum())
    mean = Fraction(s1, n) * Fraction(2) ** e0
    var = Fraction(n * s2 - s1 * s1, n * n) * Fraction(2) ** (2 * e0)
    return float(mean), math.sqrt(float(var))


STAT_LENGTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 127, 128, 129, 511, 512, 513, 65535, 65536, 65537, 200000]


def stat_families():
    """name -> function(n, rng) -> Content of one row of n samples."""
    def outlier32(n, rng):        # the first sample is the worst outlier: the one-pass shift sits far from the mean
        return Content(rows=[np.r_[np.float32(1000.123), np.full(n - 1, np.float32(1e-3))]])

    def outlier_adc(n, rng):
        return Content(counts=[np.r_[32767, np.zeros(n - 1)]], scale=0.0305, offset=0.0123)

    def dc_offset(n, rng):        # 1e4 + a few LSB of 2^-10: float32-exact, every kind
        return Content(counts=[rng.randint(-3, 4, n)], scale=2.0 ** -10, offset=1e4)

    def dc_offset_nondyadic(n, rng):
        return Content(counts=[rng.randint(-3, 4, n) + 20000], scale=0.0305, offset=0.0123)

    def constant(n, rng):
        return Content(rows=[np.full(n, np.float32(0.1))])

    def constant_adc(n, rng):
        return Content(counts=[np.full(n, 1234)], scale=-0.0305, offset=0.0123)

    def extremes_adc(n, rng):     # the int16 ends at a negative scale
        return Content(counts=[rng.choice(np.array([-32768, 32767]), n)], scale=-0.0305, offset=0.0123)

    def huge32(n, rng):           # float32 values near 3e38
        return Content(rows=[rng.uniform(2.9e38, 3.3e38, n).astype(np.float32)])

    def nonfinite(n, rng):
        r = rng.normal(60, 2, n).astype(np.float32).astype(np.float64)
        r[(n * 7) // 10] = [np.nan, np.inf, -np.inf][n % 3]
        if n % 4 == 1 and n > 3:
            r[1] = np.inf
            r[2] = -np.inf
        return Content(rows=[r])

    return dict(outlier32=outlier32, outlier_adc=outlier_adc, dc_offset=dc_offset,
                dc_offset_nondyadic=dc_offset_nondyadic, constant=constant, constant_adc=constant_adc,
                extremes_adc=extremes_adc, huge32=huge32, nonfinite=nonfinite)


def join(contents):
    if contents[0].counts is not None:
        return Content(counts=[c.counts[0] for c in contents], scale=contents[0].scale, offset=contents[0].offset)
    return Content(rows=[c.rows[0] for c in contents])


def stat_batches(make, rng):
    """The rows of STAT_LENGTHS alone (a table averaging >= 512 samples per row), and shuffled among 1000 rows of
    9 samples, so that the rows longer than 65,536 samples share warps with short ones.  Either way a row of fewer
    than 512 samples is summed by 8 lanes and a longer one by 32."""
    rows = [make(n, rng) for n in STAT_LENGTHS]
    wide = join(rows)
    mixed = rows + [make(9, rng) for _ in range(1000)]
    order = rng.permutation(len(mixed))
    narrow = join([mixed[i] for i in order])
    assert wide.lengths().sum() / len(wide.rows) >= 512 > narrow.lengths().sum() / len(narrow.rows)
    return {32: wide, 8: narrow}


def reference_stats(content):
    out = []
    for r in content.rows:
        with np.errstate(invalid="ignore", over="ignore"):
            mn, mx = np.min(r), np.max(r)
            if np.all(np.isfinite(r)):
                m, s = exact_stats(r)
            else:
                m, s = np.mean(r), np.std(r)
        out.append((m, s, mn, mx, np.max(np.abs(r))))
    return out


def check_stats(got, ref, lens, where, worst):
    for k, (m, s, mn, mx, amax) in enumerate(ref):
        gm, gs, gmn, gmx = got["mean"][k], got["std"][k], got["min"][k], got["max"][k]
        assert same_bits(np.array([gmn, gmx]), np.array([mn, mx])), (where, lens[k], gmn, mn, gmx, mx)
        if not (np.isfinite(m) and np.isfinite(s)):
            assert same_bits(np.array([gm, gs]), np.array([m, s])), (where, lens[k], gm, m, gs, s)
            continue
        if s == 0.0:
            assert gs == 0.0 and gm == m, (where, lens[k], gm, m, gs)
            continue
        dm, ds = abs(gm - m), abs(gs - s) / s
        assert dm <= 1e-12 * amax, (where, lens[k], gm, m, amax)
        if abs(m) >= 1e-3 * s:          # the relative bar where the mean is not itself lost in the spread
            assert dm <= STAT_RTOL * abs(m), (where, lens[k], gm, m, dm / abs(m))
            key = ("mean", where[0], where[2], "long" if lens[k] > 65536 else "short")
            worst[key] = max(worst.get(key, 0.0), dm / abs(m))
        assert ds <= STAT_RTOL, (where, lens[k], gs, s, ds)
        key = ("std", where[0], where[2], "long" if lens[k] > 65536 else "short")
        worst[key] = max(worst.get(key, 0.0), ds)


@pytest.fixture(scope="module")
def stat_data():
    rng = np.random.RandomState(40)
    data = {}
    for name, make in stat_families().items():
        for g, content in stat_batches(make, rng).items():
            data[name, g] = (content, reference_stats(content))
    return data


@pytest.mark.parametrize("family", sorted(stat_families()))
def test_event_stats_against_exact_reference(ctx, stat_data, family):
    """K4 over events: one pass (<= 65,536 samples, 16-byte vectors) and two passes, G = 8 and G = 32 lanes per
    row, every source kind; mean within 1e-12 max|x| and 1e-9 relative of the exact mean, std within 1e-9 of the
    exact std, min / max bitwise, NaN / inf like NumPy."""
    worst = {}
    for g in (8, 32):
        content, ref = stat_data[family, g]
        lens = content.lengths()
        for kind in content.kinds():
            put(ctx, kind, content, phase=g % 7)
            check_stats(ctx.event_stats(len(lens)), ref, lens, (family, kind, g), worst)
    print("\nK4 worst relative error %s: %s" % (family, {k: "%.2g" % v for k, v in sorted(worst.items())}))


@pytest.mark.parametrize("family", ["outlier32", "outlier_adc", "dc_offset_nondyadic", "extremes_adc"])
def test_event_stats_alignment_invariant(ctx, stat_data, family):
    """The same rows at all eight 16-byte phases: min / max bitwise equal, mean / std within 1e-13 of the row's
    scale (the larger of |mean| and std)."""
    for g in (8, 32):
        content, _ = stat_data[family, g]
        for kind in content.kinds()[:-1]:          # not flat64: packed events have one placement
            base = None
            for phase in range(8):
                put(ctx, kind, content, phase=phase)
                got = ctx.event_stats(len(content.rows))
                if base is None:
                    base = got
                    continue
                assert same_bits(got["min"], base["min"]) and same_bits(got["max"], base["max"]), (kind, phase)
                scale = np.maximum(np.abs(base["mean"]), base["std"])
                for k in ("mean", "std"):
                    d = np.abs(got[k] - base[k])
                    assert np.all(d <= 1e-13 * scale), (kind, g, phase, k, np.max(d / scale))


def test_segment_stats_against_exact_reference(ctx):
    """K4 over the segments of a split (rows = segments of the events), ADC step data at a dyadic and a
    non-dyadic scale, every source kind."""
    rng = np.random.RandomState(41)
    lens = [3000, 20000, 70001, 250000]
    cnt = []
    for n in lens:
        steps = np.repeat(rng.randint(-20000, 20000, n // 500 + 1), 500)[:n]
        cnt.append((steps + rng.normal(0, 300, n)).clip(-32768, 32767).astype(np.int16))
    worst = {}
    for scale, offset in ((2.0 ** -8, 60.0), (0.0305, 0.0123)):
        content = Content(counts=cnt, scale=scale, offset=offset)
        for kind in content.kinds():
            put(ctx, kind, content, phase=3)
            n = ctx.statsplit(100, 1000000, 10000, oracle.min_gain(prior_segments_per_second=10))
            ctx.segment_stats()
            tab = ctx.segments(n)
            rows = [content.rows[e][s:t] for e, s, t in zip(tab["event"], tab["start"], tab["end"])]
            assert len(rows) > 100
            seg = Content(rows=rows)
            check_stats(tab, reference_stats(seg), seg.lengths(), ("segments", kind, scale), worst)
    print("\nK4 segments worst relative error: %s" % {k: "%.2g" % v for k, v in sorted(worst.items())})


# ------------------------------------------------------------------------------------------- K5 filter
def oracle_filtfilt(b, a, zi, x):
    """The oracle's sequential filtfilt with exactly the b, a, zi handed to the device."""
    b, a, zi = (np.ascontiguousarray(v, np.float64).copy() for v in (b, a, zi))
    x = np.ascontiguousarray(x, np.float64)
    out = np.empty_like(x)
    f64p = ctypes.POINTER(ctypes.c_double)
    assert orc.lib().orc_filtfilt(b.ctypes.data_as(f64p), a.ctypes.data_as(f64p), zi.ctypes.data_as(f64p), len(b),
                                  x.ctypes.data_as(f64p), len(x), out.ctypes.data_as(f64p)) == 0
    return out


def filter_content(lens, rng, dyadic):
    cnt = []
    for n in lens:
        steps = np.repeat(rng.randint(-8000, 8000, n // 700 + 1), 700)[:n]
        cnt.append((steps + rng.normal(0, 600, n)).clip(-32768, 32767).astype(np.int16))
    return Content(counts=cnt, scale=2.0 ** -6, offset=60.0) if dyadic else \
        Content(counts=cnt, scale=0.0305, offset=0.0123)


def run_filter(ctx, kind, content, b, a, zi):
    put(ctx, kind, content, phase=5)
    ctx.filter_events(b, a, zi)
    lens = content.lengths()
    y = ctx.event_samples(int(lens.sum()))
    return np.split(y, np.cumsum(lens)[:-1])


@pytest.mark.parametrize("order", [3, 4, 5, 6, 7, 8])
def test_filter_sequential_orders_bitwise(ctx, order):
    """Orders 3-8 run scipy's own sequential operation order: bit for bit the oracle on every source kind."""
    rng = np.random.RandomState(50 + order)
    pad = 3 * (order + 1)
    lens = [pad + 1, pad + 2, 100, 4097, 60001]
    for fc_fs, dyadic in ((0.02, True), (0.02, False), (1e-3, True), (0.2, False)):
        b, a, zi = bessel_coefficients(order, fc_fs * 1e5, 1e5)
        content = filter_content(lens, rng, dyadic)
        refs = [oracle_filtfilt(b, a, zi, r) for r in content.rows]
        for kind in content.kinds():
            for e, y in enumerate(run_filter(ctx, kind, content, b, a, zi)):
                assert y.tobytes() == refs[e].tobytes(), (order, fc_fs, kind, lens[e])


@pytest.mark.parametrize("order", [1, 2])
def test_filter_parallel_orders_long_events_and_cutoffs(ctx, order):
    """Orders 1-2 (the parallel tiled scan): up to ~1000 tiles of 4096 samples, fc / fs from 1e-3 to 0.2;
    error <= 1e-8 of the event's largest |y| against the oracle."""
    rng = np.random.RandomState(60 + order)
    pad = 3 * (order + 1)
    lens = [pad + 1, 4095, 4097, 100003, 4000037]
    content = filter_content(lens, rng, True)
    worst = {}
    for fc_fs in (1e-3, 1e-2, 0.05, 0.2):
        b, a, zi = bessel_coefficients(order, fc_fs * 1e5, 1e5)
        refs = [oracle_filtfilt(b, a, zi, r) for r in content.rows]
        for kind in content.kinds():
            for e, y in enumerate(run_filter(ctx, kind, content, b, a, zi)):
                err = np.max(np.abs(y - refs[e])) / np.max(np.abs(refs[e]))
                key = (fc_fs, "long" if lens[e] > 100003 else "short")
                worst[key] = max(worst.get(key, 0.0), err)
                assert err <= 1e-8, (order, fc_fs, kind, lens[e], err)
    print("\nK5 order %d worst error / max|y|: %s" % (order, {k: "%.2g" % v for k, v in sorted(worst.items())}))


def test_filter_padlen_boundary_every_kind(ctx):
    """An event of exactly padlen = 3 (order + 1) samples is refused like scipy (ValueError), padlen + 1 runs."""
    rng = np.random.RandomState(70)
    for order in range(1, 9):
        b, a, zi = bessel_coefficients(order, 2000., 1e5)
        pad = 3 * (order + 1)
        ok = filter_content([pad + 1, 500], rng, True)
        short = filter_content([500, pad], rng, True)
        for kind in ok.kinds():
            put(ctx, kind, short)
            with pytest.raises(ValueError, match="padlen"):
                ctx.filter_events(b, a, zi)
            y = run_filter(ctx, kind, ok, b, a, zi)
            ref = oracle_filtfilt(b, a, zi, ok.rows[0])
            assert np.max(np.abs(y[0] - ref)) <= 1e-8 * np.max(np.abs(ref)), (order, kind)
