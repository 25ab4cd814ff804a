#!/usr/bin/env python
"""bench.py -- headline benchmark: Msamples/s segmented (threshold + SpeedyStatSplit).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c1|c2|c3|c4|c5]
                    [--dump-outputs DIR]

A step is one pass of the hot path (lambda_event_parser threshold scan + rule selection -> [Event.filter] ->
SpeedyStatSplit prefix sums / split search -> segment table -> segment statistics) over one batch of synthetic
input.  `--config` picks the BASELINE.json configuration (default c2 = configs[1], the one the metric is quoted on):

    c1  configs[0]  6 M-sample trace, 500 events                       (N > 1: one such piece per GPU, weak scaling)
    c2  configs[1]  60 M-sample trace, 5000 events                     (N > 1: one such piece per GPU, weak scaling)
    c3  configs[2]  ONE 360 M-sample trace, 30000 events               (N > 1: cut into N contiguous chunks, STRONG scaling)
    c4  configs[3]  20 events of 10 M samples, max_width = 1e6         (N > 1: whole events dealt over the GPUs, strong;
                                                                        at most 3 events per GPU at 8: a 6.67x cap)
    c5  configs[4]  1000 files of 2.5 M samples at 250 kHz, Event.filter(1, 2000) + SpeedyStatSplit, through
                    Experiment.parse(batch=FileBatch)                  (N > 1: files dealt over the GPUs, strong)

Every line carries `roofline`, `cpu_baseline` (N = 1), `e2e` (host buffers in, host tables out) and `parity` (the tables
of the run against a full-size fixture made from the reference / the CPU oracle).

`--impl reference` times the reference's own CPU code for the same path: the unmodified cparsers.pyx compiled into
oracle/_ref (falling back to the C port) plus the NumPy / scipy statements of parsers.py:148-155, DataTypes.py:270-271
and core.py:209-223, on all host cores, on a bounded sample of the same workload.
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

THRESHOLD = 110.0
RULES = dict(duration_gt=1000, min_gt=-0.5, max_lt=110.0)
DEV_RULES = dict(rule_mask=7, duration_gt=RULES["duration_gt"], duration_lt=0, min_gt=RULES["min_gt"],
                 max_lt=RULES["max_lt"])
SPLIT = dict(min_width=100, max_width=1000000, window_width=10000)
EVENTS_PER_GPU = 5000
METRIC = "Msamples/s segmented (threshold+SpeedyStatSplit)"
FS5 = 2.5e5                                  # c5: sampling rate of the files
SPLIT5 = dict(min_width=100, window_width=10000, sampling_freq=FS5, cutoff_freq=2000., prior_segments_per_second=10)
FILTER5 = (1, 2000.)

CONFIGS = {
    "c1": dict(kind="trace", events=500, seed=0, scaling="weak", steps=20,
               what="BASELINE configs[0]: synthetic 60 s 100 kHz float32 trace, 500 events (~6 M samples)"),
    "c2": dict(kind="trace", events=EVENTS_PER_GPU, seed=1, scaling="weak", steps=20,
               what="BASELINE configs[1]: synthetic 100 kHz float32 trace, 5000 events (~60 M samples)"),
    "c3": dict(kind="trace", events=30000, seed=2, scaling="strong", steps=8,
               what="BASELINE configs[2]: ONE synthetic 1 h 100 kHz float32 trace, 30000 events (~360 M samples)"),
    "c4": dict(kind="long", events=20, length=10_000_000, scaling="strong", steps=3,
               what="BASELINE configs[3]: long-event regime, 20 events of 10 M samples each (200 M samples), "
                    "SpeedyStatSplit(max_width=1e6)"),
    "c5": dict(kind="batch", files=1000, scaling="strong", steps=10,
               what="BASELINE configs[4]: batch of 1000 files of 2.49 M samples at 250 kHz (2.49 G samples), "
                    "Event.filter(order=1, cutoff=2000) + SpeedyStatSplit(prior_segments_per_second=10, "
                    "sampling_freq=2.5e5, cutoff_freq=2000) through Experiment.parse(batch=FileBatch)"),
}
PIPE = ("; lambda_event_parser(threshold=110, rules=[duration>1000, min>-0.5, max<110]) + SpeedyStatSplit(min_width=100, "
        "window_width=10000) (min_gain=-0.0) + segment stats; ADC-quantised samples (tier A)")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler(object):
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.002)

    def start(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------
# CPU reference path (timed as the baseline; never on the product path)
# --------------------------------------------------------------------------------------
def _cpu_threshold(x64, threshold):
    """lambda_event_parser.parse + _lambda_select, statement by statement (parsers.py:136-155)."""
    mask = np.where(x64 < threshold, 1, 0)
    mask = np.abs(np.diff(mask))
    tics = np.concatenate(([0], np.where(mask == 1)[0] + 1, [x64.shape[0]]))
    del mask
    pieces = [(tics[i], np.array(c)) for i, c in enumerate(np.split(x64, tics[1:-1]))]
    keep = []
    for start, cur in pieces:
        ok = np.all([cur.shape[0] > RULES["duration_gt"], np.min(cur) > RULES["min_gt"],
                     np.max(cur) < RULES["max_lt"]])
        if ok:
            keep.append((int(start), cur))
    return keep


_W = {}


def _ref_module():
    import oracle
    if _W.get("ref") is None:
        try:
            _W["ref"] = oracle.load_ref_cparsers() if oracle.ref_available() else False
        except Exception:
            _W["ref"] = False
    return _W["ref"]


def _cpu_split_events(job):
    """FastStatSplit.parse per event (after scipy's filtfilt for c5, DataTypes.py:268-271) + one read of
    mean/std/min/max per segment (BASELINE.md 3.4).  job = (events, split kwargs, filter (order, cutoff, fs) or None)."""
    import oracle
    events, kw, filt = job
    n_seg = 0
    acc = 0.0
    ref = _ref_module()
    ba = None
    if filt is not None:
        from scipy import signal
        ba = signal.bessel(filt[0], filt[1] / (filt[2] / 2.), btype='low', analog=0, output='ba')
    for cur in events:
        if ba is not None:
            from scipy import signal
            cur = signal.filtfilt(ba[0], ba[1], cur)
        if ref:
            segs = ref.FastStatSplit(**kw).parse(cur)
            for s in segs:
                c = s.current
                acc += np.mean(c) + np.std(c) + np.min(c) + np.max(c)
            n_seg += len(segs)
        else:
            bp = oracle.statsplit(cur, **kw)
            edges = np.concatenate(([0], bp, [len(cur)]))
            for a, b in zip(edges[:-1], edges[1:]):
                c = cur[a:b]
                acc += np.mean(c) + np.std(c) + np.min(c) + np.max(c)
            n_seg += len(edges) - 1
    return n_seg, acc


def cpu_reference_run(traces, cores, kw=None, filt=None):
    """One pass of the reference path over the float64 traces on `cores` processes.
    Returns (seconds, events, segments, kind)."""
    import oracle
    kw = dict(SPLIT) if kw is None else kw
    kind = "reference" if oracle.ref_available() else "port"
    t0 = time.perf_counter()
    events = []
    for x64 in traces:
        events += [cur for _, cur in _cpu_threshold(x64, THRESHOLD)]
    if cores <= 1:
        n_seg, _ = _cpu_split_events((events, kw, filt))
    else:
        # the workers are forked AFTER the events exist and read them from the parent's memory: nothing but two
        # integers per task is pickled (round 1 shipped the event arrays through the pool's pipe every step, which
        # understated the multi-core reference)
        import multiprocessing as mp
        _W["events"] = (events, kw, filt)
        with mp.get_context("fork").Pool(cores) as pool:
            n_seg = sum(pool.map(_cpu_split_slice, [(i, cores * 4) for i in range(cores * 4)]))
        _W["events"] = None
    return time.perf_counter() - t0, len(events), n_seg, kind


def _cpu_split_slice(task):
    i, stride = task
    events, kw, filt = _W["events"]
    return _cpu_split_events((events[i::stride], kw, filt))[0]


def cpu_sample(cfg, cores):
    """The bounded sample of a config's workload the CPU arm is timed on: (float64 traces, split kwargs, filter,
    description)."""
    from pypore_b200 import synth
    if cfg["kind"] == "trace":
        n = min(cfg["events"], 150 * cores if cores > 1 else 1500)
        x = synth.make_trace(n, seed=cfg["seed"], tier="A").astype(np.float64)
        return [x], dict(SPLIT), None, "%d-event prefix of the workload trace (%d samples)" % (n, len(x))
    if cfg["kind"] == "long":
        n = 1 if cores <= 1 else min(cfg["events"], max(2, cores // 4))
        x = synth.make_long_trace(n, 2_000_000, seed0=100, tier="A").astype(np.float64)
        return [x], dict(SPLIT), None, ("%d long event(s) of 2 M samples (the workload's are 10 M: same regime, a fifth "
                                        "of the length, %d samples)" % (n, len(x)))
    n = 1 if cores <= 1 else min(8, cores)
    xs = [synth.make_trace(208, seed=900 + i, tier="A").astype(np.float64) for i in range(n)]
    kw = dict(min_width=100, max_width=1000000, window_width=10000, sampling_freq=int(FS5), cutoff_freq=2000.,
              prior_segments_per_second=10)
    return xs, kw, (1, 2000., FS5), "%d of the batch's files (%d samples)" % (n, sum(len(x) for x in xs))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    traces, kw, filt, what = cpu_sample(cfg, cores)
    n = sum(len(x) for x in traces)
    for _ in range(min(args.warmup, 1)):
        cpu_reference_run([x[:len(x) // 8] for x in traces], cores, kw, filt)
    t = 0.0
    for _ in range(args.steps):
        dt, ne, ns, kind = cpu_reference_run(traces, cores, kw, filt)
        t += dt
    value = n * args.steps / t / 1e6
    sample = "%s per step, %d processes over events" % (what, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.config, args.gpus, args),
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "events": ne, "segments": ns,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_line(cfg):
    """`cpu_baseline` of the GPU arm's line: the reference as it is -- one process -- on a bounded sample."""
    traces, kw, filt, what = cpu_sample(cfg, 1)
    dt, ne, ns, kind = cpu_reference_run(traces, 1, kw, filt)
    return {"value": sum(len(x) for x in traces) / dt / 1e6, "unit": "Msamples/s", "cores": 1, "kind": kind,
            "sample": what + ", one pass, single process (the reference is single-threaded)"}


# --------------------------------------------------------------------------------------
# shared pieces of the GPU arm
# --------------------------------------------------------------------------------------
def workload_config(name, n_gpus, args):
    cfg = CONFIGS[name]
    out = {"name": name, "workload": cfg["what"] + (PIPE if cfg["kind"] != "batch" else "; ADC-quantised samples (tier A)")}
    if cfg["kind"] == "trace":
        epg = getattr(args, "events_per_gpu", None) or cfg["events"]
        if cfg["scaling"] == "weak":
            out["events_per_gpu"] = epg
            out["partition"] = ("one such trace per GPU, the pieces forming one contiguous trace cut mid-event, halo + "
                                "table all-gather" if n_gpus > 1 else "single GPU")
        else:
            out["events_total"] = epg
            out["partition"] = ("the trace cut into %d contiguous chunks, halo + table all-gather" % n_gpus
                                if n_gpus > 1 else "single GPU")
        out["l2"] = "inputs (4 B/sample trace + 16 B/event-sample prefix sums) exceed the 126 MB L2; no explicit flush"
    elif cfg["kind"] == "long":
        out["partition"] = ("whole events dealt round-robin over the GPUs (an event's window chain cannot be split), "
                            "table all-gather" if n_gpus > 1 else "single GPU")
        out["l2"] = "inputs (800 MB trace + 3.2 GB prefix sums) exceed the 126 MB L2; no explicit flush"
    else:
        out["files"] = getattr(args, "files", None) or cfg["files"]
        out["partition"] = "files dealt round-robin over the GPUs, ragged table all-gather" if n_gpus > 1 else "single GPU"
        out["l2"] = "every resident pass holds ~60 M samples (240 MB + 1 GB of float64 / prefix sums): exceeds the L2"
    return out


def parity_rows(ev_rows, seg_rows, fixture, key, what):
    """Counts + SHA-256 of the event rows (start, length) and segment rows (event, start, end) against a fixture.
    Outside every timed region; never raises."""
    try:
        g = np.load(os.path.join(ROOT, "tests", "golden", fixture), allow_pickle=False)
        names = {"c2_full.npz": ("events", "default_segments", "events_sha", "default_sha")}.get(
            fixture, (key + "events", key + "segments", key + "events_sha", key + "segments_sha"))
        if names[0] not in g.files:
            return {"error": "no fixture %s in %s" % (names[0], fixture)}
        out = {"fixture": "tests/golden/%s (%s)" % (fixture, what),
               "events": int(len(ev_rows)) if ev_rows is not None else None, "events_expected": int(g[names[0]]),
               "segments": int(len(seg_rows)), "segments_expected": int(g[names[1]]),
               "segments_bit_exact": bool(sha(np.asarray(seg_rows, np.int64)) == str(g[names[3]]))}
        if ev_rows is not None:
            out["events_bit_exact"] = bool(sha(np.asarray(ev_rows, np.int64)) == str(g[names[2]]))
        return out
    except Exception as exc:  # a reporting extra must not cost the bench line
        return {"error": "%s: %s" % (type(exc).__name__, exc)}


DUMP_BYTES = 60_000_000     # --dump-outputs: array bytes in all, so that the files with their headers stay under 64 MB


def device_tables(ctx, res):
    """The event and segment tables a step left on the device, as a caller of the pipeline reads them, in float64
    (row indices and sample positions are below 2**53: exact)."""
    ev_start, ev_len = ctx.events(res["events"])
    seg = ctx.segments(res["segments"])
    tables = {"event": {"start": ev_start, "length": ev_len},
              "segment": {k: seg[k] for k in ("event", "start", "end", "mean", "std", "min", "max")}}
    return {t: {k: np.asarray(v, np.float64) for k, v in cols.items()} for t, cols in tables.items()}


def dump_outputs(out_dir, tables):
    """Writes column k of table t as out_dir/<t>_<k>.npy.  A table larger than its share of DUMP_BYTES is cut to a
    fixed, seeded sample of its rows (the same rows for the same row count), whose indices go to <t>_row.npy."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES
    for i, (name, cols) in enumerate(tables.items()):
        n = len(next(iter(cols.values())))
        share = budget // (len(tables) - i)
        if 8 * n * len(cols) > share:
            rows = np.sort(np.random.default_rng(0).choice(n, share // (8 * (len(cols) + 1)), replace=False))
            cols = dict({k: v[rows] for k, v in cols.items()}, row=rows.astype(np.float64))
        for k, v in cols.items():
            np.save(os.path.join(out_dir, "%s_%s.npy" % (name, k)), v)
            budget -= v.nbytes


def ncu_traffic(kernel="k3_split", metrics=("dram__bytes_read.sum", "dram__bytes_write.sum")):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the newest committed `ncu --set full`
    capture of the default command (profiles/*_ncu_summary.csv), plus whether that capture is of THIS state of the
    kernels: its file name must start with the tag in profiles/CURRENT (the tag the kernels were last profiled under;
    changing a kernel without a new capture leaves the tag behind and the figure is reported as stale)."""
    import csv
    import glob
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        current = open(os.path.join(ROOT, "profiles", "CURRENT")).read().split()[0]
    except Exception:
        current = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_summary.csv")), reverse=True):
        try:
            rows = list(csv.reader(open(path)))
            col = next(i for i, n in enumerate(rows[0]) if n.startswith(kernel))
            tot = 0.0
            for r in rows:
                if r and r[0] in metrics:
                    tot += float(r[col]) * unit.get(r[1], 1.0)
            if tot > 0:
                base = os.path.basename(path)
                return tot, base, bool(current and base.startswith(current))
        except Exception:
            continue
    return None, None, False


class Timer(object):
    """K steps between two CUDA events on `stream`, bracketed by a barrier + device synchronisation, max over ranks."""

    def __init__(self, torch, dist, world, stream):
        self.torch, self.dist, self.world, self.stream = torch, dist, world, stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, fn, steps, before=None, closing=None):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        if before:
            before(steps)
        r = None
        for _ in range(steps):
            r = fn()
        if closing:
            closing()      # stream-level joins: the closing event waits for everything the steps left in flight
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, r


def split_roofline(counters_cand, split_ms, kernel, bound, note, use_traffic):
    peak, peak_src = peaks()
    split_bytes = 16.0 * counters_cand
    gbs = split_bytes / (split_ms / 1e3) / 1e9
    traffic, src, fresh = ncu_traffic(kernel) if use_traffic else (None, None, False)
    return {"bound": bound, "kernel": kernel, "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
            "traffic": traffic, "traffic_source": src, "traffic_stale": (not fresh) if traffic else None,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": split_bytes, "note": note}


K3_NOTE = ("algorithmic bytes = one 16 B {c,c2} pair per candidate evaluation (SURVEY 8d).  The bound is NOT HBM: the "
           "prefix sums are re-read from L2 once per recursion level (DRAM traffic is a third of the algorithmic bytes) "
           "and the kernel is bound by instruction issue and dependent latency -- ~0.6 warp instructions per cycle and "
           "scheduler (issue_frac; instruction count from the ncu capture named beside it) -- see DESIGN.md 4")


def init_dist(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    if world > 1:
        # a job smaller than the node takes GPUs from both halves of the board (both sockets' upload bandwidth)
        from pypore_b200.dist import device_for_rank
        local = device_for_rank(local, torch.cuda.device_count())
    torch.cuda.set_device(local)
    if world > 1:
        # one process per GPU: stay on the cores (and host memory) next to this GPU's PCIe root
        from pypore_b200.dist import bind_near_gpu
        bound = bind_near_gpu(local)
        if os.environ.get("PYPORE_B200_BENCH_VERBOSE"):
            print("rank %d bound to %d cores" % (rank, bound), file=sys.stderr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return torch, dist, world, rank, local


def base_line(args, cfg, world, value, ms, e2e_value, h2d, d2h, launches, clocks):
    return {"metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.config, world, args),
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": clocks}


# --------------------------------------------------------------------------------------
# c1 / c2 / c3: one trace (or one contiguous chunk of it per GPU)
# --------------------------------------------------------------------------------------
def run_trace(args):
    torch, dist, world, rank, local = init_dist(args)
    from pypore_b200 import _lib, synth
    from pypore_b200.parsers import statsplit_min_gain
    cfg = CONFIGS[args.config]
    mw, MW, W, gain = statsplit_min_gain(**SPLIT)
    ctx = _lib.Context(local)
    if args.split_kernel is not None:
        ctx.set_split_kernel(args.split_kernel == "flow")
    # every kernel, copy-stream join and collective of a step is ordered on the context's stream:
    # the timing events are recorded there
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=torch.device("cuda", local))
    timer = Timer(torch, dist, world, stream)

    # ---- synthetic input ---------------------------------------------------------------
    epg = args.events_per_gpu or cfg["events"]
    full = epg == cfg["events"]
    shard = whole = None
    if world == 1:
        x = synth.make_trace(epg, seed=cfg["seed"], tier="A")
    else:
        from pypore_b200 import dist as ppdist
        if cfg["scaling"] == "weak":
            x = ppdist.synthetic_chunk(rank, world, epg, seed0=cfg["seed"])
        else:   # one fixed trace, cut into `world` contiguous chunks wherever the cut falls
            whole = synth.make_trace(epg, seed=cfg["seed"], tier="A")
            x = np.ascontiguousarray(whole[len(whole) * rank // world:len(whole) * (rank + 1) // world])
        shard = ppdist.ShardedPipeline(ctx, rank, world)
    n_local = len(x)
    xp = torch.from_numpy(x).pin_memory().numpy()

    inflight = {"ticket": None, "last": None}

    def step_resident():
        if shard is None:
            return ctx.pipeline(THRESHOLD, min_width=mw, max_width=MW, window_width=W, min_gain=gain,
                                with_stats=True, **DEV_RULES)
        # step i+1 is enqueued before the result records of step i are read: the device never waits for the host;
        # drain_resident() reads the last step's records inside the timed region
        t = shard.step_async(THRESHOLD, DEV_RULES, mw, MW, W, gain)
        if inflight["ticket"] is not None:
            inflight["last"] = shard.finish(inflight["ticket"])
        inflight["ticket"] = t
        return inflight["last"]

    def drain_resident():
        if shard is not None and inflight["ticket"] is not None:
            inflight["last"] = shard.finish(inflight["ticket"])
            inflight["ticket"] = None
        return inflight["last"]

    last_download = {}
    # Multi-GPU end to end: the upload of step i+1 (the context's copy stream, into a second device buffer) runs
    # under step i's kernels and collectives, and the copy-out of step i's tables (a side stream, the other PCIe
    # direction) under both.  Every step's H2D and D2H are inside the timed region.
    e2e = {"remaining": 0, "loaded": False, "x": xp, "queued": 0}

    def step_e2e():
        if shard is None:
            # public host-memory entry point (pp_pipeline_host_tables): chunked H2D copy overlapped with the stages;
            # the event / segment rows a chunk has finalised are written into page-locked host tables while the
            # next chunk is still on its way, so the call returns with the whole result in host memory
            r = ctx.pipeline(THRESHOLD, min_width=mw, max_width=MW, window_width=W, min_gain=gain,
                             with_stats=True, host_trace=e2e["x"], export=True, **DEV_RULES)
            assert len(r["segment_table"]["mean"]) == r["segments"]
            return r
        if not e2e["loaded"]:
            shard.load(e2e["x"])               # first step of a run: nothing was prefetched for it
            e2e["queued"] = 0
        e2e["remaining"] -= 1
        e2e["loaded"] = e2e["remaining"] > 0
        while e2e["queued"] < min(2, e2e["remaining"]):
            shard.prefetch(e2e["x"])           # the traces of the next two steps are on their way (or queued behind
            e2e["queued"] += 1                 # the running copy) before this step runs
        r = shard.step(THRESHOLD, DEV_RULES, mw, MW, W, gain)
        if not os.environ.get("PYPORE_B200_BENCH_NO_DOWNLOAD"):   # (development switch: invalid e2e)
            # every GPU holds the whole result; it reaches host memory once, the way the trace went up: every rank's
            # process reads the rows of its own chunk over its own link (PYPORE_B200_BENCH_RANK0_DOWNLOAD: rank 0 pulls
            # the whole table instead).  The copy-out is enqueued on a side stream and collected before the next one
            # is started; finish_e2e() collects the last one.
            own = not os.environ.get("PYPORE_B200_BENCH_RANK0_DOWNLOAD")
            if own or rank == 0:
                if last_download.get("pending") is not None:
                    last_download["tables"] = last_download["pending"].wait()
                last_download["pending"] = shard.download_async(own_rows=own)
        if e2e["loaded"]:
            shard.swap()
            e2e["queued"] -= 1
        return r

    def finish_e2e():
        if shard is not None and last_download.get("pending") is not None:
            last_download["tables"] = last_download["pending"].wait()
            last_download["pending"] = None

    def arm_e2e(steps):
        e2e["remaining"], e2e["loaded"] = steps, False

    def closing():
        if shard is not None:
            drain_resident()   # (resident loop) the last step's records are read inside the timed region
            shard.wait()   # the last step's asynchronous table all-gather belongs to the timed region, and so does
            shard.join()   # the copy-out of its tables on the side stream: the closing event waits for both

    if shard is None:
        ctx.upload_trace(xp)
    else:
        shard.load(xp)
    for _ in range(max(args.warmup, 3)):
        step_resident()
    drain_resident()
    sampler = ClockSampler(local)
    launches0 = ctx.launch_count
    sampler.start()
    ms, res = timer.run(step_resident, args.steps, closing=closing)
    res = drain_resident() if shard is not None else res
    dumped = device_tables(ctx, res) if args.dump_outputs else None
    launches = ctx.launch_count - launches0
    stage = ctx.stage_ms() if shard is None else dict(shard.stage_ms)
    counters = ctx.split_counters()
    # split-kernel duration averaged over a few more steps (CUDA events inside the library, on the launch stream);
    # the clock sampler keeps polling through them -- same load -- so that a short timed region still yields samples
    split_ms = []
    k = 0
    while k < min(args.steps, 5) or (world == 1 and len(sampler.samples) < 8 and k < 200):  # ranks stay in step
        step_resident()
        drain_resident()
        split_ms.append(ctx.stage_ms()["split"] if shard is None else shard.stage_ms["split"])
        k += 1
    split_ms = float(np.mean(split_ms))
    clocks = sampler.stop()

    # End to end, the chunks need not be equal: the GPUs of a node do not get equal shares of the host's upload
    # bandwidth when all of them copy at once (on the 8 x B200 box GPUs 0-3 get 23 GB/s each, GPUs 4-7 36 GB/s).
    # The rates are measured, the SAME global trace is cut in proportion to them, and every upload ends at the same
    # time.  Results are global tables, so the parity fixture is the same.
    e2e_cut = None
    chunk_cache = {}

    def all_ranks(value):
        mine = torch.tensor([value], dtype=torch.float64, device="cuda")
        out = torch.empty(world, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(out, mine)
        return out.cpu().numpy()

    def cut_by(rates):
        """This rank's chunk of the global trace when the shares follow `rates` (same array on every rank)."""
        lens = np.asarray(shard.lens0, np.int64)
        offs = np.concatenate(([0], np.cumsum(lens)))
        cuts = ppdist.proportional_cuts(int(offs[-1]), rates)
        a, b = int(cuts[rank]), int(cuts[rank + 1])
        if cfg["scaling"] == "weak":
            def other(q):
                if q not in chunk_cache:
                    chunk_cache[q] = ppdist.synthetic_chunk(q, world, epg, seed0=cfg["seed"])
                return chunk_cache[q]
            xe = ppdist.recut_chunk(rank, cuts, lens, x, other)
        else:
            xe = whole[a:b]
        e2e["x"] = torch.from_numpy(np.ascontiguousarray(xe)).pin_memory().numpy()
        return [int(v) for v in np.diff(cuts)]

    if shard is not None and not args.even_cut:
        shard.lens0 = np.array(shard.lens)       # the even cut's chunk lengths: where the global trace's pieces lie
        rates = ppdist.measure_upload_rates(ctx, xp, dist, torch.device("cuda", local), world)
        if args.upload_rates:
            rates = np.array([float(v) for v in args.upload_rates.split(",")])[:world] * 1e9
        e2e_cut = {"upload_GBps_all_ranks_at_once": [round(4e-9 * r, 1) for r in rates], "cut": "even"}
        if rates.max() > 1.1 * rates.min():          # (same rates on every rank: same decision)
            per_rank = cut_by(rates)
            e2e_cut["cut"] = "proportional to the measured rates"
            e2e_cut["samples_per_rank"] = per_rank
    chunk_cache.clear()
    whole = None

    arm_e2e(2)
    for _ in range(2):
        step_e2e()
    finish_e2e()
    ms_e2e, res_e2e = timer.run(step_e2e, args.steps, before=arm_e2e, closing=closing)
    finish_e2e()

    upload_ms = [round(float(v), 3) for v in all_ranks(ctx.prefetch_ms())] if shard is not None else None

    # the floor under the end-to-end number on this box: every rank's upload alone (all ranks at once, nothing else
    # in flight), same page-locked buffer, same copy call
    def step_upload():
        ctx.upload_trace_async(e2e["x"], extra_capacity=0 if shard is None else shard.HALO_CAPACITY)
    ms_h2d, _ = timer.run(step_upload, min(args.steps, 5))
    ms_h2d /= min(args.steps, 5)
    if shard is not None:
        shard.load(e2e["x"])

    totals = torch.tensor([n_local, res["events"], res["segments"], res["event_samples"]], device="cuda",
                          dtype=torch.float64)
    if world > 1:
        totals = torch.tensor([shard.n_owned, res["events"], res["segments"], res["event_samples"]],
                              device="cuda", dtype=torch.float64)
        dist.all_reduce(totals)
    n_total, ev_total, seg_total, evs_total = [int(v) for v in totals.tolist()]

    if rank == 0:
        peak, _ = peaks()
        sec = ms / 1e3 / args.steps
        sec_e2e = ms_e2e / 1e3 / args.steps
        b_floor = 4.0 * n_total + 56.0 * seg_total + 24.0 * ev_total
        # SURVEY 8d's second figure, the reference's data flow: threshold reads N, the prefix kernel reads N_ev and
        # writes {c, c2}, the search touches one pair per candidate, statistics re-read N_ev, 56 B per segment row
        # (candidates are counted on rank 0; every rank holds a like share of the workload)
        b_alg = 4.0 * n_total + 20.0 * evs_total + 16.0 * counters["candidates"] * world + 4.0 * evs_total + 56.0 * seg_total
        line = base_line(args, cfg, world, n_total / sec / 1e6, ms, n_total / sec_e2e / 1e6, 4 * n_total,
                         56 * seg_total + 16 * ev_total + 160 * world, launches, clocks)
        line["e2e"]["ms_per_step"] = ms_e2e / args.steps
        line["e2e"]["h2d_only_ms_per_step"] = ms_h2d
        line["e2e"]["h2d_only_note"] = ("the uploads of all %d ranks alone, at once: %.1f GB/s of host-to-device copy "
                                        "on this box; the end-to-end step cannot be shorter" %
                                        (world, 4.0 * n_total / ms_h2d / 1e6))
        if e2e_cut is not None:
            e2e_cut["upload_ms_per_rank_last_step"] = upload_ms
            line["e2e"]["chunks"] = e2e_cut
        line["roofline"] = split_roofline(counters["candidates"], split_ms, "k3_split", "issue", K3_NOTE,
                                          world == 1 and args.config == "c2" and full)
        # warp instructions of the profiled launch (smsp__inst_executed.sum of the newest committed capture, taken on
        # configs[1]: 240.4 M candidates) scale with the candidate count; 148 SMs x 4 schedulers x 1 issue per cycle
        inst, inst_src, inst_fresh = ncu_traffic("k3_split", ("smsp__inst_executed.sum",))
        inst = inst or 617e6
        line["roofline"]["issue_frac"] = (inst / 240.4e6 * counters["candidates"]) / (148 * 4 * 1.965e9 * split_ms / 1e3)
        line["roofline"]["warp_instructions_per_launch_c2"] = inst
        line["roofline"]["warp_instructions_source"] = inst_src
        line["roofline"]["warp_instructions_stale"] = not inst_fresh
        line["pipeline_roofline"] = {
            "b_floor_bytes": b_floor, "achieved": b_floor / sec / 1e9 / world, "peak": peak, "unit": "GB/s per GPU",
            "frac": b_floor / sec / 1e9 / world / peak, "b_alg_bytes": b_alg,
            "achieved_b_alg": b_alg / sec / 1e9 / world, "frac_b_alg": b_alg / sec / 1e9 / world / peak,
            "note": "north-star figure: B_floor = 4 N + 56 S + 24 E over the step; the >= 60 % target is not met under "
                    "either definition (the split search evaluates 4 candidates per trace sample)"}
        line["stage_ms"], line["split_ms"] = stage, split_ms
        line["counts"] = {"samples": n_total, "events": ev_total, "event_samples": evs_total, "segments": seg_total,
                          "candidates_rank0": counters["candidates"]}
        if shard is not None:
            line["host_planned_fallback_steps"] = int(shard.fallbacks)
        if full:
            if shard is None:
                es, el = res_e2e["event_table"]
                t = res_e2e["segment_table"]
                ev_rows = np.stack([np.asarray(es, np.int64), np.asarray(el, np.int64)], axis=1)
                seg_rows = np.stack([np.asarray(t["event"]).astype(np.int64), np.asarray(t["start"], np.int64),
                                     np.asarray(t["end"], np.int64)], axis=1)
            else:
                t = shard.download()          # (outside the timed regions) the whole table, for the hash
                ev_rows = np.stack([np.asarray(t["ev_start"], np.int64), np.asarray(t["ev_len"], np.int64)], axis=1)
                seg_rows = np.stack([np.asarray(t[k], np.int64) for k in ("seg_event", "seg_start", "seg_end")], axis=1)
            if args.config == "c2":
                line["parity"] = (parity_rows(ev_rows, seg_rows, "c2_full.npz", "", "real reference, full size")
                                  if world == 1 else
                                  parity_rows(ev_rows, seg_rows, "sharded_full.npz", "w%d_" % world,
                                              "CPU oracle on the uncut trace, full size; hashes equal the real reference's, "
                                              "tests/golden/reference_full_check.json"))
            elif args.config == "c1" and world == 1:
                line["parity"] = parity_rows(ev_rows, seg_rows, "bench_configs.npz", "c1_", "real reference, full size")
            elif args.config == "c3":
                line["parity"] = parity_rows(ev_rows, seg_rows, "bench_configs.npz", "c3_",
                                             "CPU oracle on the uncut 360 M-sample trace; hashes equal the real reference's, "
                                             "tests/golden/reference_full_check.json")
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_line(cfg)
        print(json.dumps(line), flush=True)
    if dumped:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


# --------------------------------------------------------------------------------------
# c4: long events, whole events per GPU
# --------------------------------------------------------------------------------------
def run_long(args):
    torch, dist, world, rank, local = init_dist(args)
    from pypore_b200 import _lib, synth
    from pypore_b200.parsers import statsplit_min_gain
    cfg = CONFIGS["c4"]
    n_events = args.long_events or cfg["events"]
    mw, MW, W, gain = statsplit_min_gain(**SPLIT)
    ctx = _lib.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=torch.device("cuda", local))
    timer = Timer(torch, dist, world, stream)
    mine = list(range(rank, n_events, world))           # global event ids of this rank, round-robin
    if world == 1:
        x = synth.make_long_trace(n_events, cfg["length"], seed0=100, tier="A")     # the fixture's trace itself
    else:
        rng = np.random.RandomState(100 + 7919 + 1000 * (rank + 1))
        parts = []
        for e in mine:
            parts.append(synth.quantise(rng.normal(synth.OPEN_MEAN, synth.OPEN_STD, 4000)))
            parts.append(synth.make_long_event(cfg["length"], 100 + e, "A"))
        parts.append(synth.quantise(rng.normal(synth.OPEN_MEAN, synth.OPEN_STD, 4000)))
        x = np.concatenate(parts)
    xp = torch.from_numpy(x).pin_memory().numpy()
    tables = {}

    state = {"pack": None}

    def exchange(r):
        """Every rank's event and segment rows on every GPU, without leaving the device: the result records are
        all-gathered (8 words per rank), pp_pack_tables writes this rank's rows (event ids offset by the event counts of
        the ranks before it), one all-gather moves the packed rows.  Returns (gathered [world, pad], records)."""
        from pypore_b200 import dist as ppdist
        rec = torch.tensor([0, r["events"], r["event_samples"], r["segments"], 0, 0, 0, 0], dtype=torch.int64,
                           device="cuda")
        allr = torch.empty(world * 8, dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(allr, rec)
        counts = allr.view(world, 8)[:, [1, 3]].cpu().numpy()
        pad = (int(max(2 * e + ppdist.SEG_WORDS * sg for e, sg in counts)) + 65) & ~1
        if state["pack"] is None or state["pack"].shape[0] < pad:
            state["pack"] = torch.empty(pad, dtype=torch.int64, device="cuda")
        ctx.pack_tables(allr.data_ptr(), rank, 0, state["pack"].data_ptr(), pad)
        g = ppdist.gather_packed_raw(state["pack"], pad, dist)
        return g, allr, counts

    def step(host):
        if host:
            # one chunk: the search of a 10 M-sample event cannot start before its last sample has arrived, and the
            # window chains of different events must run side by side -- a chunked upload would walk them a chunk's
            # worth (one or two events) at a time
            r = ctx.pipeline(THRESHOLD, min_width=mw, max_width=MW, window_width=W, min_gain=gain, with_stats=True,
                             host_trace=xp, chunk_samples=len(xp), **DEV_RULES)
        else:
            r = ctx.pipeline(THRESHOLD, min_width=mw, max_width=MW, window_width=W, min_gain=gain, with_stats=True,
                             **DEV_RULES)
        if world > 1:
            with torch.cuda.stream(stream):
                g, allr, counts = exchange(r)
                tables["gathered"] = (g, allr, counts)
                if host:
                    # end to end: every rank's process reads the rows of its own events into page-locked memory
                    tables["own"] = ctx.unpack_tables(g.data_ptr(), world, g.shape[1], allr.data_ptr(),
                                                      int(counts[rank][0]), int(counts[rank][1]), ranks=(rank, rank + 1))
        elif host:
            seg = ctx.segments(r["segments"], pinned=True)
            tables["ev"] = ctx.events(r["events"])
            tables["seg_int"] = np.stack([seg["event"].astype(np.int64), seg["start"], seg["end"]], axis=1)
        return r

    def merged_segment_rows():
        """(outside the timed regions, rank 0) the whole gathered table with the events' round-robin ids, sorted."""
        g, allr, counts = tables["gathered"]
        cols = ctx.unpack_tables(g.data_ptr(), world, g.shape[1], allr.data_ptr(), int(counts[:, 0].sum()),
                                 int(counts[:, 1].sum()))
        e_base = np.concatenate(([0], np.cumsum(counts[:, 0])))
        owner = np.searchsorted(e_base, cols["seg_event"], side="right") - 1        # rank that produced the row
        event = owner + world * (cols["seg_event"] - e_base[owner])                 # dealt round-robin
        rows = np.stack([event, cols["seg_start"], cols["seg_end"]], axis=1).astype(np.int64)
        return rows[np.lexsort((rows[:, 1], rows[:, 0]))]

    ctx.upload_trace(xp)
    for _ in range(max(min(args.warmup, 3), 1)):
        step(False)
    sampler = ClockSampler(local)
    launches0 = ctx.launch_count
    sampler.start()
    ms, res = timer.run(lambda: step(False), args.steps)
    dumped = device_tables(ctx, res) if args.dump_outputs else None
    launches = ctx.launch_count - launches0
    stage = ctx.stage_ms()
    counters = ctx.split_counters()
    clocks = sampler.stop()
    step(True)
    ms_e2e, res = timer.run(lambda: step(True), args.steps)
    tot = torch.tensor([len(x), res["events"], res["segments"], counters["candidates"]], device="cuda",
                       dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot)
    n_total, ev_total, seg_total, cand_total = [int(v) for v in tot.tolist()]
    if rank == 0:
        sec, sec_e2e = ms / 1e3 / args.steps, ms_e2e / 1e3 / args.steps
        line = base_line(args, cfg, world, n_total / sec / 1e6, ms, n_total / sec_e2e / 1e6, 4 * n_total,
                         56 * seg_total + 16 * ev_total, launches, clocks)
        line["roofline"] = split_roofline(
            counters["candidates"], stage["split"], "k3_spine", "latency",
            "an event's windows form a dependent chain (the next window starts at the split the current one finds): "
            "~7,650 dependent scans per 10 M-sample event, each walked by a 4-CTA cluster; the chain's latency bounds the "
            "kernel, not bandwidth.  8-GPU speed-up is capped at 20/3 = 6.67x (3 events on the busiest GPU)", False)
        line["stage_ms"] = stage
        line["counts"] = {"samples": n_total, "events": ev_total, "segments": seg_total, "candidates": cand_total}
        if n_events == cfg["events"]:
            ev_rows = np.stack(tables["ev"], axis=1) if world == 1 else None
            if world > 1:
                tables["seg_int"] = merged_segment_rows()
            line["parity"] = parity_rows(ev_rows, tables["seg_int"], "bench_configs.npz", "c4_",
                                         "CPU oracle, all 20 events; hashes equal the real reference's, tests/golden/"
                                         "reference_full_check.json" + ("" if world == 1 else "; segment rows only: event "
                                                                        "starts are rank-local when events are dealt out"))
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_line(cfg)
        print(json.dumps(line), flush=True)
    if dumped:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


# --------------------------------------------------------------------------------------
# c5: a batch of files through Experiment.parse(batch=FileBatch)
# --------------------------------------------------------------------------------------
def run_batch(args):
    torch, dist, world, rank, local = init_dist(args)
    from pypore_b200 import _lib, synth
    from pypore_b200.DataTypes import Experiment, File, bessel_coefficients
    from pypore_b200.batch import FileBatch
    from pypore_b200.parsers import RuleSet, SpeedyStatSplit, lambda_event_parser
    cfg = CONFIGS["c5"]
    n_files = args.files or cfg["files"]
    host = _lib.Context(local)
    distinct = []
    for i in range(8):       # eight distinct files, reused cyclically (the fixture's; a batch of 1000 distinct ones
        x = synth.make_trace(208, seed=900 + i, tier="A")     # would cost minutes of generation and 10 GB of host memory)
        p = host.pinned_empty(x.shape[0], np.float32)
        p[:] = x
        distinct.append(p)
    traces = [distinct[i % 8] for i in range(n_files)]
    n_total = sum(len(t) for t in traces)
    det = lambda_event_parser(threshold=110, rules=RuleSet(**RULES))
    seg = SpeedyStatSplit(**SPLIT5)
    batch = FileBatch(device=local, workers=4, rank=rank, world=world)
    timer = Timer(torch, dist, world, torch.cuda.current_stream())

    def step_e2e():
        # the reference's own call for a batch (DataTypes.py:956-988), files in page-locked host memory in, the
        # metadata tables of every file in host memory out; wall clock, because the passes run on worker streams
        exp = Experiment([File(current=t, timestep=1000. / FS5) for t in traces])
        exp.parse(event_detector=det, segmenter=seg, filter_params=FILTER5, verbose=False, meta=True, batch=batch)
        return exp

    # device-resident leg: ~26 files (64 M samples) sit behind each other on the device (one +inf sample between
    # neighbours, what a grouped pass of FileBatch holds) and the whole pipeline incl. the Bessel filter runs on them
    group = []
    used = 0
    for t in traces:
        if used + len(t) + 1 > (1 << 26):
            break
        group.append(t)
        used += len(t) + 1
    resident = np.concatenate([np.concatenate((t, np.array([np.inf], np.float32))) for t in group])[:-1]
    host.upload_trace(resident)
    mw, MW, W, gain = seg._params()
    filt = bessel_coefficients(FILTER5[0], FILTER5[1], FS5)
    rs_stream = torch.cuda.ExternalStream(host.stream_handle, device=torch.device("cuda", local))
    rtimer = Timer(torch, dist, world, rs_stream)

    def step_resident():
        return host.pipeline(THRESHOLD, min_width=mw, max_width=MW, window_width=W, min_gain=gain, filter_ba=filt,
                             with_stats=True, **DEV_RULES)
    for _ in range(3):
        step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = host.launch_count
    ms_res, res = rtimer.run(step_resident, args.steps)
    dumped = device_tables(host, res) if args.dump_outputs else None
    launches = host.launch_count - launches0
    stage = host.stage_ms()
    counters = host.split_counters()
    step_e2e()                                   # warm-up batch: every worker context's buffers grown
    timer.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        exp = step_e2e()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.stop()
    if world > 1:
        tt = torch.tensor([t_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e2e = float(tt.item())
    if rank == 0:
        tb = exp.tables
        value = len(resident) * world / (ms_res / 1e3 / args.steps) / 1e6
        line = base_line(args, cfg, world, value, ms_res, n_total / (t_e2e / args.steps) / 1e6,
                         4 * n_total, 56 * tb.n_segments + 48 * tb.n_events, launches, clocks)
        line["value_note"] = ("device-resident leg: one grouped pass of %d files (%d samples) per GPU, whole pipeline "
                              "incl. the Bessel filtfilt, CUDA events; e2e: the %d-file batch through "
                              "Experiment.parse(batch=FileBatch), host wall clock around the call"
                              % (len(group), len(resident), n_files))
        line["roofline"] = split_roofline(counters["candidates"], stage["split"], "k3_split", "issue", K3_NOTE, False)
        line["stage_ms"] = stage
        line["counts"] = {"samples": n_total, "files": n_files, "events": tb.n_events, "segments": tb.n_segments}
        e8, s8 = tb.file_rows(7)[0][1], tb.file_rows(7)[1][1]         # rows of the first eight files = the fixture's batch
        ev_rows = np.stack([tb.events[k][:e8] for k in ("file", "start", "length")], axis=1)
        seg_rows = np.stack([tb.segments[k][:s8] for k in ("file", "event", "start", "end")], axis=1)
        par = parity_rows(ev_rows, seg_rows, "c5_files.npz", "psps10_", "CPU oracle: scipy-equivalent filtfilt + split, the "
                          "eight distinct files of the batch; hashes equal the real reference's, tests/golden/"
                          "reference_full_check.json")
        per_file = np.bincount(tb.segments["file"], minlength=n_files)
        par["every_file_like_its_template"] = bool(all(per_file[i] == per_file[i % 8] for i in range(n_files)))
        line["parity"] = par
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_line(cfg)
        print(json.dumps(line), flush=True)
    if dumped:
        dump_outputs(args.dump_outputs, dumped)
    batch.close()
    host.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--events-per-gpu", type=int, default=None,
                    help="development: a smaller c1/c2/c3 workload (no parity fixture then)")
    ap.add_argument("--long-events", type=int, default=None, help="development: fewer c4 events")
    ap.add_argument("--files", type=int, default=None, help="development: fewer c5 files")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--upload-rates", default=None, help="development: relative upload rates per rank, e.g. 1,1.5")
    ap.add_argument("--even-cut", action="store_true",
                    help="N > 1, end to end: equal chunks per GPU instead of chunks proportional to the measured upload rates")
    ap.add_argument("--split-kernel", default=None, choices=["flow", "level"],
                    help="development: force k3_flow / k3_split (default: the library's default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the event and segment tables of the last one as DIR/<name>.npy "
                         "(float64; a fixed, seeded sample of the rows above 64 MB), to compare two builds output for "
                         "output; one GPU and --impl ours only")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = CONFIGS[args.config]["steps"] if args.impl == "ours" else 3
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours and --gpus 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        {"trace": run_trace, "long": run_long, "batch": run_batch}[CONFIGS[args.config]["kind"]](args)


if __name__ == "__main__":
    main()
