"""int16 ADC counts against float32 / float64 input on one GPU, c2 workload (bench.py's trace: 59,883,057 samples of
tier A, i.e. k/32 with |k| < 2^15).  One JSON line.

    python scripts/adc_e2e.py [--warmup 3] [--steps 20] [--out profiles/adc_e2e_line.json]

Arms, alternated inside every step so that they share the machine's state:
  e2e_f32 / e2e_adc      pipeline(host_trace=..., export=True) from page-locked memory: the float32 trace against
                         AdcTrace(round(x * 32), 1/32, 0), which decodes to exactly the same values
  copy_f32 / copy_adc    the bare host-to-device copy of the trace (240 MB against 120 MB, page-locked, CUDA events)
  resident_f32 / _adc    pipeline on the resident trace, with pp_stage_ms per stage
  real_f64 / real_adc    a real amplifier's scale (counts * 0.0305 + 0.0123, not float32-representable): today's
                         float64-trace route (whole upload at 8 B per sample, resident pipeline, table download)
                         against pipeline(host_trace=AdcTrace, export=True); plus the resident prefix stage and the
                         strict-order redo count (n_seq_redo) of both
Step times are host clocks around calls that end in a device synchronise.  The c2 arms' tables are hashed against
tests/golden/c2_full.npz (the real reference's), the real-scale ADC tables against the float64 route's.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pypore_b200 import _lib, synth  # noqa: E402
from pypore_b200.adc import AdcTrace  # noqa: E402
from pypore_b200.parsers import statsplit_min_gain  # noqa: E402

RULES = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
REAL = (0.0305, 0.0123)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def table_sha(ev, seg):
    es, el = ev
    rows = np.stack([np.asarray(seg["event"]).astype(np.int64), np.asarray(seg["start"], np.int64),
                     np.asarray(seg["end"], np.int64)], axis=1)
    return sha(np.stack([np.asarray(es, np.int64), np.asarray(el, np.int64)], axis=1)), sha(rows)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def stats(v):
    v = np.asarray(v)
    return dict(median_ms=round(float(np.median(v)), 4), mean_ms=round(float(v.mean()), 4),
                min_ms=round(float(v.min()), 4), max_ms=round(float(v.max()), 4), n=int(len(v)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "adc_e2e_line.json"))
    a = ap.parse_args()
    info = gpu_info()
    gain = statsplit_min_gain(**SPLIT)[3]
    kw = dict(min_gain=gain, **SPLIT, **RULES)
    g = np.load(os.path.join(ROOT, "tests", "golden", "c2_full.npz"))
    want_c2 = (str(g["events_sha"]), str(g["default_sha"]))

    x = synth.make_trace(5000, seed=1, tier="A")
    n = len(x)
    ctx = _lib.Context(0)
    x32 = ctx.pinned_empty(n, np.float32)
    x32[:] = x
    c2 = ctx.pinned_empty(n, np.int16)
    c2[:] = np.round(x.astype(np.float64) * 32)
    t2 = AdcTrace(c2, 1.0 / 32, 0.0)
    assert np.array_equal(t2.decode(), x.astype(np.float64))
    cr = ctx.pinned_empty(n, np.int16)
    cr[:] = np.round((x.astype(np.float64) - REAL[1]) / REAL[0])
    tr = AdcTrace(cr, *REAL)
    x64 = ctx.pinned_empty(n, np.float64)
    x64[:] = tr.decode()

    src32 = torch.from_numpy(x).pin_memory()
    src16 = torch.from_numpy(c2.copy()).pin_memory()
    dst32 = torch.empty(n, dtype=torch.float32, device="cuda")
    dst16 = torch.empty(n, dtype=torch.int16, device="cuda")

    def copy_ms(dst, src):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src, non_blocking=True)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        ctx.sync()
        return (time.perf_counter() - t0) * 1e3, r

    def e2e(trace):
        return timed(lambda: ctx.pipeline(110.0, host_trace=trace, export=True, **kw))

    def resident(upload):
        upload()
        ms, r = timed(lambda: ctx.pipeline(110.0, **kw))
        return ms, r, ctx.stage_ms(), ctx.split_counters()

    def real_f64():
        def run():
            ctx.upload_trace_f64(x64)
            r = ctx.pipeline(110.0, **kw)
            return ctx.events(r["events"]), ctx.segments(r["segments"])
        return timed(run)

    times = {k: [] for k in ("e2e_f32", "e2e_adc", "copy_f32", "copy_adc", "resident_f32", "resident_adc",
                             "real_f64", "real_adc")}
    stage = {k: [] for k in ("resident_f32", "resident_adc", "real_f64", "real_adc")}
    counters, parity = {}, {}
    for step in range(a.warmup + a.steps):
        keep = step >= a.warmup
        last = step == a.warmup + a.steps - 1
        for name, fn in (("e2e_f32", lambda: e2e(x32)), ("e2e_adc", lambda: e2e(t2))):
            ms, r = fn()
            if keep:
                times[name].append(ms)
            if last:
                parity[name] = table_sha(r["event_table"], r["segment_table"]) == want_c2
        if keep:
            times["copy_f32"].append(copy_ms(dst32, src32))
            times["copy_adc"].append(copy_ms(dst16, src16))
        for name, up in (("resident_f32", lambda: ctx.upload_trace(x32)), ("resident_adc", lambda: ctx.upload_trace_adc16(t2)),
                         ("real_f64", lambda: ctx.upload_trace_f64(x64)), ("real_adc", lambda: ctx.upload_trace_adc16(tr))):
            ms, r, st, cnt = resident(up)
            if keep:
                stage[name].append(st)
                if name.startswith("resident"):
                    times[name].append(ms)
            counters[name] = cnt
        ms, (ev64, seg64) = real_f64()
        if keep:
            times["real_f64"].append(ms)
        ms, r = e2e(tr)
        if keep:
            times["real_adc"].append(ms)
        if last:
            parity["real_adc_vs_f64"] = table_sha(r["event_table"], r["segment_table"]) == table_sha(ev64, seg64)
            parity["real_events"], parity["real_segments"] = int(r["events"]), int(r["segments"])

    line = dict(
        what="c2 trace (%d samples, 5000 events) as float32 / int16 ADC counts / float64 current, one GPU" % n,
        gpu=info, warmup=a.warmup, steps=a.steps,
        times={k: stats(v) for k, v in times.items()},
        stage_ms={k: {s: round(float(np.median([d[s] for d in v])), 4) for s in _lib.STAGES} for k, v in stage.items()},
        prefix_ms={k: round(float(np.median([d["prefix"] for d in stage[k]])), 4) for k in ("real_f64", "real_adc")},
        n_seq_redo={k: counters[k]["seq_redo"] for k in counters},
        bytes_per_sample=dict(f32=4, adc=2, f64=8),
        parity=parity,
        timing="host clock around calls ending in a device synchronise; copies: CUDA events around one "
               "page-locked host-to-device copy",
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line))
    ok = parity["e2e_f32"] and parity["e2e_adc"] and parity["real_adc_vs_f64"]
    ctx.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
