"""HMM decode times on one GPU: c2 (5000 events, ~306 k segments) and one c4-style event.

    python scripts/hmm_bench.py --out profiles/hmm_c2_line.json

c2: the c2 trace goes through the resident pipeline (threshold scan -> SpeedyStatSplit -> statistics); the step is
timed with the host clock around pp_pipeline, which ends in a synchronise.  Each decode (Viterbi / forward at
S = 8, 32, 64, 128, Viterbi with the merge) is timed with CUDA events on the context stream after a warm-up; a
merge changes the table, so the pipeline runs again (untimed) before every merged decode.
c4-style: one 10 M-sample event, SpeedyStatSplit(max_width=1e6); torch.profiler splits the Viterbi decode into
the forward kernel and the traceback.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pypore_b200 import _lib, synth  # noqa: E402
from pypore_b200.hmm import HMM  # noqa: E402
from pypore_b200.parsers import SpeedyStatSplit  # noqa: E402

STATES = (8, 32, 64, 128)
REPS = 10


def model(S, seed=0):
    rng = np.random.default_rng(seed)
    trans = rng.uniform(0.0, 1.0, (S, S)) + 4 * np.eye(S)
    return HMM(np.sort(rng.uniform(0.0, 110.0, S)), rng.uniform(1.0, 6.0, S), trans, ends=rng.uniform(0, 0.5, S))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def timed(ctx, fn, reps):
    s = torch.cuda.ExternalStream(ctx.stream_handle)
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        fn()
        e1.record(s)
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def kernel_ms(ctx, fn):
    """Device time per kernel name of one call of fn (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        ctx.sync()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.key.startswith("_Z") or "hmm" in ev.key or "k3c" in ev.key or "k4_" in ev.key:
            out[ev.key] = out.get(ev.key, 0.0) + ev.device_time_total / 1e3
    return out


def stat(v):
    v = sorted(v)
    return dict(median=v[len(v) // 2], min=v[0], max=v[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hmm_c2_line.json"))
    args = ap.parse_args()
    ctx = _lib.Context(0)
    line = dict(gpu=gpu_info(), what=__doc__.split("\n\n")[0].strip())

    # ---- c2 ----
    x = synth.make_trace(5000, seed=1, tier="A")
    mw, MW, W, gain = SpeedyStatSplit(min_width=100, window_width=10000)._params()
    kw = dict(rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0, min_width=mw, max_width=MW,
              window_width=W, min_gain=gain)
    ctx.upload_trace(x)

    def pipeline():
        return ctx.pipeline(110, **kw)

    for _ in range(3):
        counts = pipeline()
    step = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        pipeline()
        step.append((time.perf_counter() - t0) * 1e3)
    line["c2"] = dict(samples=int(x.shape[0]), events=counts["events"], segments=counts["segments"],
                      pipeline_step_ms=stat(step), decode_ms={})
    for S in STATES:
        m = model(S, S)
        row = {}
        for algorithm in ("viterbi", "forward"):
            timed(ctx, lambda: ctx.hmm_decode(m, algorithm), 2)
            row[algorithm] = stat(timed(ctx, lambda: ctx.hmm_decode(m, algorithm), REPS))
        merged = []
        for _ in range(REPS + 1):
            pipeline()
            merged += timed(ctx, lambda: ctx.hmm_decode(m, "viterbi", merge=True), 1)
        row["viterbi_merge"] = stat(merged[1:])
        pipeline()
        row["merged_segments"] = ctx.hmm_decode(m, "viterbi", merge=True)
        pipeline()
        row["kernels_viterbi_ms"] = kernel_ms(ctx, lambda: ctx.hmm_decode(m, "viterbi"))
        line["c2"]["decode_ms"]["S%d" % S] = row
        print(json.dumps({"S": S, **{k: v for k, v in row.items() if k != "kernels_viterbi_ms"}}), flush=True)

    # ---- c4-style: one 10 M-sample event ----
    ev = synth.make_long_event(10_000_000, seed=100, tier="A").astype(np.float64)
    mw, MW, W, gain = SpeedyStatSplit(max_width=1000000)._params()
    ctx.upload_events_f64([ev])
    t0 = time.perf_counter()
    n_seg = ctx.statsplit(mw, MW, W, gain)
    ctx.segment_stats()
    ctx.sync()
    split_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    n_seg = ctx.statsplit(mw, MW, W, gain)
    ctx.segment_stats()
    ctx.sync()
    split_ms = min(split_ms, (time.perf_counter() - t0) * 1e3)
    c4 = dict(samples=int(ev.shape[0]), segments=n_seg, split_and_stats_ms=split_ms, decode_ms={})
    for S in STATES:
        m = model(S, S)
        timed(ctx, lambda: ctx.hmm_decode(m, "viterbi"), 1)
        total = stat(timed(ctx, lambda: ctx.hmm_decode(m, "viterbi"), 3))
        k = kernel_ms(ctx, lambda: ctx.hmm_decode(m, "viterbi"))
        tb = sum(v for name, v in k.items() if "traceback" in name)
        fw = sum(v for name, v in k.items() if "k_hmm_warp" in name or "k_hmm_cta" in name)
        c4["decode_ms"]["S%d" % S] = dict(viterbi=total, forward_kernel_ms=fw, traceback_ms=tb,
                                          traceback_share=tb / (tb + fw) if tb + fw > 0 else None)
        print(json.dumps({"c4_S": S, **c4["decode_ms"]["S%d" % S]}), flush=True)
    line["c4_style"] = c4
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(line, fh, indent=1)
    print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    main()
