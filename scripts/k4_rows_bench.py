"""K4 (k4_segment_stats) alone on tables of short rows, long rows and a mix: segment and event statistics of c2's
trace (rows ~130 / ~8,000 samples), of a c5-style 250 kHz batch (Event.filter(1, 2000) + prior_segments_per_second
= 10: long segments) and of c4-style 10 M-sample events (event rows taking two passes).  One JSON line per table.

    python scripts/k4_rows_bench.py [reps=30]

Times are CUDA events on the context's stream around one launch (segment statistics: the `stats` stage of
pp_segment_stats; event statistics: pp_event_stats_download, i.e. the launch plus the copy of four 8-byte columns
per event), median over `reps` calls after one warm-up.  Select another build with PYPORE_B200_LIB to compare."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pypore_b200 import _lib, synth  # noqa: E402
from pypore_b200.DataTypes import bessel_coefficients  # noqa: E402
from pypore_b200.parsers import statsplit_min_gain  # noqa: E402

RULES = dict(threshold=110.0, rule_mask=7, duration_gt=1000, duration_lt=0, min_gt=-0.5, max_lt=110.0)


def timed(ctx, stream, fn, reps):
    fn()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def table(ctx, stream, name, x, split, filt, reps):
    ctx.upload_trace(x)
    mw, MW, W, gain = statsplit_min_gain(**split)
    r = ctx.pipeline(min_width=mw, max_width=MW, window_width=W, min_gain=gain, filter_ba=filt, **RULES)
    ne, ns = r["events"], r["segments"]
    seg = ctx.segments(ns, stats=False)
    seg_len = (seg["end"] - seg["start"]).astype(np.float64)
    stats = []
    for _ in range(reps):
        ctx.segment_stats()
        ctx.sync()
        stats.append(ctx.stage_ms()["stats"])
    line = dict(table=name, events=ne, segments=ns, event_samples=r["event_samples"],
                segment_rows_ge_512=float(np.mean(seg_len >= 512)), mean_segment=float(seg_len.mean()),
                segment_stats_ms=float(np.median(stats)),
                event_stats_ms=timed(ctx, stream, lambda: ctx.event_stats(ne), reps),
                gpu=torch.cuda.get_device_name(0), lib=os.environ.get("PYPORE_B200_LIB") or "in-tree")
    print(json.dumps(line), flush=True)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    ctx = _lib.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=torch.device("cuda", 0))
    table(ctx, stream, "c2", synth.make_trace(5000, seed=1, tier="A"),
          dict(min_width=100, max_width=1000000, window_width=10000), None, reps)
    fs = 2.5e5
    table(ctx, stream, "c5_batch_of_8_files", synth.make_trace(8 * 208, seed=900, tier="A"),
          dict(min_width=100, window_width=10000, sampling_freq=fs, cutoff_freq=2000., prior_segments_per_second=10),
          bessel_coefficients(1, 2000., fs), reps)
    table(ctx, stream, "c4_20_events", synth.make_long_trace(20, 10000000),
          dict(min_width=100, max_width=1000000, window_width=10000), None, max(reps // 3, 3))
    ctx.close()


if __name__ == "__main__":
    main()
