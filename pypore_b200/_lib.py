"""ctypes binding of libpypore_b200.so (include/pypore_b200.h).

There is no CPU fallback: if the CUDA library is missing or no B200-class device
is present, importing works (so CPU-only tooling can introspect the package) but
the first compute call raises.
"""
import ctypes
import os

import numpy as np

from .adc import AdcTrace

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PYPORE_B200_LIB") or os.path.join(HERE, "libpypore_b200.so")  # override: development variants only

PP_OK = 0
PP_ERR_CUDA, PP_ERR_ARG, PP_ERR_CAPACITY, PP_ERR_STATE, PP_ERR_FILTER_LEN = -1, -2, -3, -4, -5
RULE_DURATION_GT, RULE_MIN_GT, RULE_MAX_LT, RULE_DURATION_LT = 1, 2, 4, 8
PREFIX_AUTO, PREFIX_SEQUENTIAL, PREFIX_PARALLEL = 0, 1, 2
STAGES = ("threshold", "select", "filter", "prefix", "split", "compact", "stats")

_c = ctypes
_i64 = _c.c_int64
_f64p = _c.POINTER(_c.c_double)
_f32p = _c.POINTER(_c.c_float)
_i64p = _c.POINTER(_c.c_int64)
_i32p = _c.POINTER(_c.c_int32)
_u8p = _c.POINTER(_c.c_uint8)


class PipelineParams(_c.Structure):
    _fields_ = [
        ("threshold", _c.c_double),
        ("rule_mask", _c.c_int),
        ("duration_gt", _i64), ("duration_lt", _i64),
        ("min_gt", _c.c_double), ("max_lt", _c.c_double),
        ("filter_ncoef", _c.c_int),
        ("filter_b", _f64p), ("filter_a", _f64p), ("filter_zi", _f64p),
        ("min_width", _c.c_int), ("max_width", _c.c_int), ("window_width", _c.c_int),
        ("min_gain", _c.c_double),
        ("prefix_mode", _c.c_int),
        ("with_stats", _c.c_int),
    ]


class HostTables(_c.Structure):
    """pp_host_tables: page-locked host buffers pp_pipeline_host_tables fills chunk by chunk."""
    _fields_ = [
        ("cap_events", _i64), ("ev_start", _c.c_void_p), ("ev_len", _c.c_void_p),
        ("cap_segments", _i64), ("seg_event", _c.c_void_p), ("seg_start", _c.c_void_p), ("seg_end", _c.c_void_p),
        ("mean", _c.c_void_p), ("std", _c.c_void_p), ("min", _c.c_void_p), ("max", _c.c_void_p),
    ]


class UnpackedTables(_c.Structure):
    """pp_unpacked_tables: one array per column of the gathered multi-GPU result."""
    _fields_ = [("cap_events", _i64), ("cap_segments", _i64), ("ev_start", _c.c_void_p), ("ev_len", _c.c_void_p),
                ("seg_event", _c.c_void_p), ("seg_start", _c.c_void_p), ("seg_end", _c.c_void_p),
                ("mean", _c.c_void_p), ("std", _c.c_void_p), ("min", _c.c_void_p), ("max", _c.c_void_p)]


class Hmm(_c.Structure):
    """pp_hmm: a model in log space (pypore_b200.hmm.HMM builds it)."""
    _fields_ = [("n_states", _c.c_int), ("mean", _f64p), ("inv_std", _f64p), ("log_norm", _f64p),
                ("log_start", _f64p), ("log_trans", _f64p), ("log_end", _f64p)]


HMM_ALGORITHMS = {"viterbi": 0, "forward": 1}

# name -> (restype, argtypes); every symbol include/pypore_b200.h declares
SIGNATURES = {
    "pp_version": (_c.c_int, []),
    "pp_device_count": (_c.c_int, []),
    "pp_create": (_c.c_int, [_c.c_int, _c.c_void_p, _c.POINTER(_c.c_void_p)]),
    "pp_destroy": (None, [_c.c_void_p]),
    "pp_last_error": (_c.c_char_p, [_c.c_void_p]),
    "pp_sync": (_c.c_int, [_c.c_void_p]),
    "pp_set_option": (_c.c_int, [_c.c_void_p, _c.c_int, _i64]),
    "pp_get_option": (_c.c_int, [_c.c_void_p, _c.c_int, _i64p]),
    "pp_launch_count": (_i64, [_c.c_void_p]),
    "pp_stage_ms": (_c.c_int, [_c.c_void_p, _c.c_int, _c.POINTER(_c.c_float)]),
    "pp_trace_upload": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _i64]),
    "pp_trace_upload_f64": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64]),
    "pp_trace_upload_adc16": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _c.c_double, _c.c_double]),
    "pp_adc16_check": (_c.c_int, [_c.c_double, _c.c_double]),
    "pp_adc16_key_threshold": (_c.c_int, [_c.c_double, _c.c_double, _c.c_double, _i32p, _i32p]),
    "pp_trace_prefetch": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _i64]),
    "pp_trace_swap": (_c.c_int, [_c.c_void_p]),
    "pp_trace_adopt": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _i64]),
    "pp_trace_append": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _c.c_int]),
    "pp_trace_truncate": (_c.c_int, [_c.c_void_p, _i64]),
    "pp_trace_len": (_i64, [_c.c_void_p]),
    "pp_trace_device_ptr": (_c.c_void_p, [_c.c_void_p]),
    "pp_threshold_scan": (_c.c_int, [_c.c_void_p, _c.c_double, _i64, _i64p]),
    "pp_runs_download": (_c.c_int, [_c.c_void_p, _i64, _i64p, _i64p, _f64p, _f64p, _u8p]),
    "pp_runs_download_range": (_c.c_int, [_c.c_void_p, _i64, _i64, _i64p, _i64p, _f64p, _f64p, _u8p]),
    "pp_select_events": (_c.c_int, [_c.c_void_p, _c.c_int, _i64, _i64, _c.c_double, _c.c_double,
                                    _c.c_int, _c.c_int, _i64p, _i64p]),
    "pp_set_events": (_c.c_int, [_c.c_void_p, _i64p, _i64p, _i64]),
    "pp_append_event": (_c.c_int, [_c.c_void_p, _i64, _i64]),
    "pp_events_download": (_c.c_int, [_c.c_void_p, _i64, _i64p, _i64p]),
    "pp_events_upload_f64": (_c.c_int, [_c.c_void_p, _f64p, _i64p, _i64]),
    "pp_filter_events": (_c.c_int, [_c.c_void_p, _f64p, _f64p, _f64p, _c.c_int]),
    "pp_event_samples_download": (_c.c_int, [_c.c_void_p, _i64, _f64p]),
    "pp_statsplit": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _c.c_int, _i64p]),
    "pp_segment_stats": (_c.c_int, [_c.c_void_p]),
    "pp_segments_download": (_c.c_int, [_c.c_void_p, _i64, _i32p, _i64p, _i64p, _f64p, _f64p, _f64p, _f64p]),
    "pp_event_stats_download": (_c.c_int, [_c.c_void_p, _i64, _f64p, _f64p, _f64p, _f64p]),
    "pp_table_device_ptr": (_c.c_void_p, [_c.c_void_p, _c.c_int]),
    "pp_split_counters": (_c.c_int, [_c.c_void_p, _i64p]),
    "pp_debug_screen": (_c.c_int, [_c.c_void_p, _i64, _c.c_int, _c.c_int, _c.c_int, _f64p, _f64p, _u8p, _f64p]),
    "pp_debug_prefix": (_c.c_int, [_c.c_void_p, _i64, _f64p, _f64p, _u8p]),
    "pp_debug_lg2_error": (_c.c_int, [_c.c_void_p, _f64p]),
    "pp_stream": (_c.c_void_p, [_c.c_void_p]),
    "pp_trace_prefetch_ms": (_c.c_int, [_c.c_void_p, _c.POINTER(_c.c_float)]),
    "pp_host_alloc": (_c.c_int, [_c.c_void_p, _i64, _c.POINTER(_c.c_void_p)]),
    "pp_host_free": (None, [_c.c_void_p, _c.c_void_p]),
    "pp_prefix": (_c.c_int, [_c.c_void_p, _c.c_int]),
    "pp_window_gains": (_c.c_int, [_c.c_void_p, _i64, _c.c_int, _i32p, _i32p, _c.c_int, _f64p, _i64]),
    "pp_shard_scan": (_c.c_int, [_c.c_void_p, _c.c_double, _i64, _c.c_void_p]),
    "pp_shard_finish": (_c.c_int, [_c.c_void_p, _c.POINTER(PipelineParams), _c.c_int, _c.c_int, _c.c_int, _i64, _i64,
                                   _c.c_void_p]),
    "pp_shard_commit": (_c.c_int, [_c.c_void_p, _i64p]),
    "pp_shard_plan": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.POINTER(PipelineParams), _i64,
                                 _c.c_void_p]),
    "pp_shard_finish_planned": (_c.c_int, [_c.c_void_p, _c.POINTER(PipelineParams), _c.c_void_p, _c.c_void_p]),
    "pp_trace_extend": (_c.c_int, [_c.c_void_p, _i64]),
    "pp_pack_tables": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _i64, _c.c_void_p, _i64]),
    "pp_ctl_create": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.POINTER(_c.c_void_p)]),
    "pp_ctl_open": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.POINTER(_c.c_void_p)]),
    "pp_ctl_exchange": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p]),
    "pp_unpack_tables": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _i64, _c.c_void_p, _c.POINTER(UnpackedTables),
                                    _c.c_int, _c.c_void_p]),
    "pp_unpack_tables_range": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _i64, _c.c_void_p, _c.c_int, _c.c_int,
                                          _c.POINTER(UnpackedTables), _c.c_int, _c.c_void_p]),
    "pp_pipeline_host": (_c.c_int, [_c.c_void_p, _f32p, _i64, _i64, _c.POINTER(PipelineParams), _i64p]),
    "pp_pipeline_host_tables": (_c.c_int, [_c.c_void_p, _f32p, _i64, _i64, _c.POINTER(PipelineParams),
                                           _c.POINTER(HostTables), _i64p]),
    "pp_pipeline_host_adc16": (_c.c_int, [_c.c_void_p, _c.c_void_p, _i64, _c.c_double, _c.c_double, _i64,
                                          _c.POINTER(PipelineParams), _c.POINTER(HostTables), _i64p]),
    "pp_pipeline": (_c.c_int, [_c.c_void_p, _c.POINTER(PipelineParams), _i64p]),
    "pp_hmm_decode": (_c.c_int, [_c.c_void_p, _c.POINTER(Hmm), _c.c_int, _c.c_int, _i64p]),
    "pp_hmm_decode_sequences": (_c.c_int, [_c.c_void_p, _c.POINTER(Hmm), _c.c_int, _f64p, _i64p, _i64]),
    "pp_hmm_download": (_c.c_int, [_c.c_void_p, _i64, _f64p, _i64, _i32p]),
}

_lib = None


class PyPoreCudaError(RuntimeError):
    pass


def load():
    """Load the shared library and attach signatures.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PyPoreCudaError(
            "libpypore_b200.so is not built (run `python -m pypore_b200.build`); "
            "pypore_b200 has no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _ptr(a, typ):
    return a.ctypes.data_as(typ) if a is not None else None


class Context(object):
    """One pp_ctx: a device, a stream and the resident trace / tables."""

    def __init__(self, device=0, stream=None):
        self._L = load()
        h = _c.c_void_p()
        r = self._L.pp_create(int(device), _c.c_void_p(stream) if stream else None, _c.byref(h))
        if r != PP_OK or not h:
            raise PyPoreCudaError(
                "pp_create(device=%d) failed (code %d): a CUDA device of compute capability 10.x "
                "(B200) is required; there is no CPU fallback" % (device, r))
        self._h = h
        if os.environ.get("PYPORE_B200_SPLIT_KERNEL"):   # development: flow | level
            self._L.pp_set_option(h, 3, 1 if os.environ["PYPORE_B200_SPLIT_KERNEL"] == "flow" else 0)
        self.device = int(device)
        self._keep = []  # host arrays that must outlive async copies

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_arena", None):
                self._L.pp_host_free(self._h, self._arena[0])
                self._arena = None
            for p, _cap in getattr(self, "_table_arenas", {}).values():
                self._L.pp_host_free(self._h, p)
            self._table_arenas = {}
            for p in getattr(self, "_pinned_keep", []):   # pinned_empty() arrays die with the context
                self._L.pp_host_free(self._h, p)
            self._pinned_keep = []
            self._L.pp_destroy(self._h)
            self._h = None

    def pinned_empty(self, n, dtype):
        """A new page-locked numpy array (freed with the context); for traces given to
        pipeline(host_trace=...) so that the chunked copy really is asynchronous."""
        dtype = np.dtype(dtype)
        p = _c.c_void_p()
        nbytes = max(int(n) * dtype.itemsize, 1)
        self._ck(self._L.pp_host_alloc(self._h, nbytes, _c.byref(p)))
        self._pinned_keep = getattr(self, "_pinned_keep", [])
        self._pinned_keep.append(p.value)
        buf = (_c.c_char * nbytes).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(n))

    def _arena_views(self, spec):
        """Views (name -> array) laid out back to back in the context's grow-only pinned arena.
        Valid until the next pinned download on this context."""
        total = sum(((n * np.dtype(dt).itemsize + 63) // 64) * 64 for _, n, dt in spec) + 64
        arena = getattr(self, "_arena", None)
        if arena is None or arena[1] < total:
            if arena is not None:
                self._L.pp_host_free(self._h, arena[0])
            p = _c.c_void_p()
            cap = int(total * 1.25)
            self._ck(self._L.pp_host_alloc(self._h, cap, _c.byref(p)))
            self._arena = arena = (p.value, cap)
        out, off = {}, 0
        for name, n, dt in spec:
            nbytes = n * np.dtype(dt).itemsize
            buf = (_c.c_char * max(nbytes, 1)).from_address(arena[0] + off)
            out[name] = np.frombuffer(buf, dtype=dt, count=n)
            off += ((nbytes + 63) // 64) * 64
        return out

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, r):
        if r == PP_OK:
            return
        msg = self._L.pp_last_error(self._h)
        msg = msg.decode("utf-8", "replace") if msg else ""
        if r == PP_ERR_FILTER_LEN:
            raise ValueError(msg)
        if r == PP_ERR_ARG:
            raise ValueError("pypore_b200: " + msg)
        raise PyPoreCudaError("pypore_b200 error %d: %s" % (r, msg))

    # -- trace ---------------------------------------------------------------
    def upload_trace(self, x32, extra_capacity=0):
        x32 = np.ascontiguousarray(x32, dtype=np.float32)
        self._keep = [x32]
        self._ck(self._L.pp_trace_upload(self._h, x32.ctypes.data, x32.shape[0], int(extra_capacity)))
        self.sync()  # pageable host memory: do not return before the copy has consumed it
        self._keep = []
        return x32.shape[0]

    def upload_trace_f64(self, x64):
        """A float64 trace, kept as float64 on the device (pp_trace_upload_f64)."""
        x64 = np.ascontiguousarray(x64, dtype=np.float64)
        self._keep = [x64]
        self._ck(self._L.pp_trace_upload_f64(self._h, x64.ctypes.data, x64.shape[0]))
        self.sync()
        self._keep = []
        return x64.shape[0]

    def upload_trace_adc16(self, trace):
        """An AdcTrace, kept as int16 counts on the device (pp_trace_upload_adc16)."""
        self._keep = [trace.counts]
        self._ck(self._L.pp_trace_upload_adc16(self._h, trace.counts.ctypes.data, len(trace), trace.scale,
                                               trace.offset))
        self.sync()
        self._keep = []
        return len(trace)

    def upload_trace_async(self, x32, extra_capacity=0):
        """For pinned host arrays; caller keeps `x32` alive until sync()."""
        assert x32.dtype == np.float32 and x32.flags.c_contiguous
        self._keep = [x32]
        self._ck(self._L.pp_trace_upload(self._h, x32.ctypes.data, x32.shape[0], int(extra_capacity)))

    def prefetch_ms(self):
        """Duration of the copy that brought up the trace swap_trace() made resident last (waits for it)."""
        ms = _c.c_float()
        self._ck(self._L.pp_trace_prefetch_ms(self._h, _c.byref(ms)))
        return float(ms.value)

    def prefetch_trace(self, x32, extra_capacity=0):
        """Start the upload of the NEXT trace (pinned float32 array; the caller keeps it alive until swap_trace()
        has been followed by a sync) while the resident one is being processed."""
        assert x32.dtype == np.float32 and x32.flags.c_contiguous
        self._keep_next = (getattr(self, "_keep_next", None) or [])[-2:] + [x32]
        self._ck(self._L.pp_trace_prefetch(self._h, x32.ctypes.data, x32.shape[0], int(extra_capacity)))

    def swap_trace(self):
        """The prefetched trace becomes the resident one (stream-level wait for its copy)."""
        self._ck(self._L.pp_trace_swap(self._h))
        self._keep = [getattr(self, "_keep_next", None)]

    def adopt_trace(self, dev_ptr, n, capacity=None):
        self._ck(self._L.pp_trace_adopt(self._h, _c.c_void_p(int(dev_ptr)), int(n), int(capacity or n)))

    def append_trace(self, src_ptr, n, src_is_device):
        self._ck(self._L.pp_trace_append(self._h, _c.c_void_p(int(src_ptr)), int(n), int(bool(src_is_device))))

    def truncate_trace(self, n):
        self._ck(self._L.pp_trace_truncate(self._h, int(n)))

    def extend_trace(self, n):
        """`n` samples were written by the caller directly after the trace end (halo received in place)."""
        self._ck(self._L.pp_trace_extend(self._h, int(n)))

    @property
    def trace_len(self):
        return int(self._L.pp_trace_len(self._h))

    @property
    def trace_ptr(self):
        return self._L.pp_trace_device_ptr(self._h)

    def sync(self):
        self._ck(self._L.pp_sync(self._h))

    @property
    def stream_handle(self):
        """cudaStream_t of the context as an integer (for torch.cuda.ExternalStream)."""
        return int(self._L.pp_stream(self._h) or 0)

    def set_option(self, option, value):
        self._ck(self._L.pp_set_option(self._h, int(option), int(value)))

    def get_option(self, option):
        v = _i64()
        self._ck(self._L.pp_get_option(self._h, int(option), _c.byref(v)))
        return int(v.value)

    def set_screening(self, on):
        """Two-stage split search (default on); off = exact arithmetic for every candidate."""
        self.set_option(0, 1 if on else 0)

    def set_spine_kernel(self, on):
        """Long events walked by the 1024-thread spine kernel first (default on); off = by the work-queue CTAs."""
        self.set_option(1, 1 if on else 0)

    def set_split_ctas(self, n):
        """Persistent CTAs of the split search (0 = one full wave).  Same tables for any value; contexts that share
        a GPU take a fraction of a wave each (batch.FileBatch)."""
        self.set_option(2, int(n))

    def set_split_kernel(self, flow):
        """Split search kernel: True = k3_flow (independent warps, no barriers), False = k3_split (level-synchronous
        CTAs).  Same tables either way."""
        self.set_option(3, 1 if flow else 0)

    @property
    def launch_count(self):
        return int(self._L.pp_launch_count(self._h))

    def stage_ms(self):
        out = {}
        ms = _c.c_float()
        for i, name in enumerate(STAGES):
            self._ck(self._L.pp_stage_ms(self._h, i, _c.byref(ms)))
            out[name] = float(ms.value)
        return out

    # -- K1 ------------------------------------------------------------------
    def threshold_scan(self, threshold, scan_len=-1):
        n = _i64()
        self._ck(self._L.pp_threshold_scan(self._h, float(threshold), int(scan_len), _c.byref(n)))
        return int(n.value)

    def runs(self, n_runs):
        start = np.empty(n_runs, np.int64)
        length = np.empty(n_runs, np.int64)
        mn = np.empty(n_runs, np.float64)
        mx = np.empty(n_runs, np.float64)
        below = np.empty(n_runs, np.uint8)
        self._ck(self._L.pp_runs_download(self._h, n_runs, _ptr(start, _i64p), _ptr(length, _i64p),
                                          _ptr(mn, _f64p), _ptr(mx, _f64p), _ptr(below, _u8p)))
        return start, length, mn, mx, below.astype(bool)

    def runs_range(self, first, count):
        start = np.empty(count, np.int64)
        length = np.empty(count, np.int64)
        mn = np.empty(count, np.float64)
        mx = np.empty(count, np.float64)
        below = np.empty(count, np.uint8)
        self._ck(self._L.pp_runs_download_range(self._h, int(first), int(count), _ptr(start, _i64p),
                                                _ptr(length, _i64p), _ptr(mn, _f64p), _ptr(mx, _f64p),
                                                _ptr(below, _u8p)))
        return start, length, mn, mx, below.astype(bool)

    def select_events(self, rule_mask, duration_gt=0, duration_lt=0, min_gt=0.0, max_lt=0.0,
                      skip_first=False, skip_last=False):
        ne, ns = _i64(), _i64()
        self._ck(self._L.pp_select_events(self._h, int(rule_mask), int(duration_gt), int(duration_lt),
                                          float(min_gt), float(max_lt), int(skip_first), int(skip_last),
                                          _c.byref(ne), _c.byref(ns)))
        return int(ne.value), int(ns.value)

    def set_events(self, start, length):
        start = np.ascontiguousarray(start, np.int64)
        length = np.ascontiguousarray(length, np.int64)
        self._ck(self._L.pp_set_events(self._h, _ptr(start, _i64p), _ptr(length, _i64p), start.shape[0]))

    def append_event(self, start, length):
        self._ck(self._L.pp_append_event(self._h, int(start), int(length)))

    def events(self, n_events):
        start = np.empty(n_events, np.int64)
        length = np.empty(n_events, np.int64)
        self._ck(self._L.pp_events_download(self._h, n_events, _ptr(start, _i64p), _ptr(length, _i64p)))
        return start, length

    def upload_events_f64(self, arrays):
        lens = np.asarray([a.shape[0] for a in arrays], np.int64)
        flat = np.ascontiguousarray(np.concatenate(arrays) if len(arrays) > 1 else arrays[0], np.float64)
        self._ck(self._L.pp_events_upload_f64(self._h, _ptr(flat, _f64p), _ptr(lens, _i64p), lens.shape[0]))
        return lens

    # -- K5 ------------------------------------------------------------------
    def filter_events(self, b, a, zi):
        b = np.ascontiguousarray(b, np.float64)
        a = np.ascontiguousarray(a, np.float64)
        zi = np.ascontiguousarray(zi, np.float64)
        self._ck(self._L.pp_filter_events(self._h, _ptr(b, _f64p), _ptr(a, _f64p), _ptr(zi, _f64p), b.shape[0]))

    def event_samples(self, n_samples):
        out = np.empty(n_samples, np.float64)
        self._ck(self._L.pp_event_samples_download(self._h, n_samples, _ptr(out, _f64p)))
        return out

    # -- K2..K4 --------------------------------------------------------------
    def statsplit(self, min_width, max_width, window_width, min_gain, prefix_mode=PREFIX_AUTO):
        n = _i64()
        self._ck(self._L.pp_statsplit(self._h, int(min_width), int(max_width), int(window_width),
                                      float(min_gain), int(prefix_mode), _c.byref(n)))
        return int(n.value)

    def prefix(self, prefix_mode=PREFIX_AUTO):
        self._ck(self._L.pp_prefix(self._h, int(prefix_mode)))

    def window_gains(self, ev, ps, pe, min_width):
        """Exact gains of every candidate of the windows [ps[w], pe[w]) of event `ev` (list of arrays)."""
        ps = np.ascontiguousarray(ps, np.int32)
        pe = np.ascontiguousarray(pe, np.int32)
        n = np.maximum(pe.astype(np.int64) - ps - 2 * int(min_width) + 1, 0)
        out = np.empty(int(n.sum()), np.float64)
        self._ck(self._L.pp_window_gains(self._h, int(ev), ps.shape[0], _ptr(ps, _i32p), _ptr(pe, _i32p),
                                         int(min_width), _ptr(out, _f64p), out.shape[0]))
        return np.split(out, np.cumsum(n)[:-1])

    def segment_stats(self):
        self._ck(self._L.pp_segment_stats(self._h))

    def segments(self, n_segments, stats=True, pinned=False):
        """Segment table as numpy arrays.  pinned=True returns views of the context's page-locked
        arena (full-rate D2H copy, no extra host copy); they are overwritten by the next pinned download."""
        if pinned:
            spec = [("event", n_segments, np.int32), ("start", n_segments, np.int64), ("end", n_segments, np.int64)]
            if stats:
                spec += [(k, n_segments, np.float64) for k in ("mean", "std", "min", "max")]
            out = self._arena_views(spec)
            ev, start, end = out["event"], out["start"], out["end"]
        else:
            ev = np.empty(n_segments, np.int32)
            start = np.empty(n_segments, np.int64)
            end = np.empty(n_segments, np.int64)
            out = {"event": ev, "start": start, "end": end}
            if stats:
                for k in ("mean", "std", "min", "max"):
                    out[k] = np.empty(n_segments, np.float64)
        self._ck(self._L.pp_segments_download(
            self._h, n_segments, _ptr(ev, _i32p), _ptr(start, _i64p), _ptr(end, _i64p),
            _ptr(out.get("mean"), _f64p), _ptr(out.get("std"), _f64p), _ptr(out.get("min"), _f64p),
            _ptr(out.get("max"), _f64p)))
        return out

    def event_stats(self, n_events):
        out = {k: np.empty(n_events, np.float64) for k in ("mean", "std", "min", "max")}
        self._ck(self._L.pp_event_stats_download(self._h, n_events, _ptr(out["mean"], _f64p),
                                                 _ptr(out["std"], _f64p), _ptr(out["min"], _f64p),
                                                 _ptr(out["max"], _f64p)))
        return out

    def table_ptr(self, which):
        return self._L.pp_table_device_ptr(self._h, int(which))

    def split_counters(self):
        out = np.zeros(8, np.int64)
        self._ck(self._L.pp_split_counters(self._h, _ptr(out, _i64p)))
        return dict(candidates=int(out[0]), scans=int(out[1]), seq_redo=int(out[2]), tasks=int(out[3]),
                    exact=int(out[4]), sure=int(out[5]), multi=int(out[6]), full=int(out[7]))

    def debug_screen(self, ev, ps, pe, min_width):
        n = pe - ps - 2 * min_width + 1
        hs, he, ok = np.empty(n), np.empty(n), np.empty(n, np.uint8)
        eps = _c.c_double()
        self._ck(self._L.pp_debug_screen(self._h, int(ev), int(ps), int(pe), int(min_width), _ptr(hs, _f64p),
                                         _ptr(he, _f64p), _ptr(ok, _u8p), _c.byref(eps)))
        return hs, he, ok.astype(bool), float(eps.value)

    def debug_prefix(self, n_events, n_samples):
        """The resident prefix sums (c = cumsum(x), c2 = cumsum(x*x), flat event space) and, per event, whether
        the strict-order kernel computed them."""
        cap = max(int(n_events), int(n_samples))
        c, c2, redone = np.empty(cap), np.empty(cap), np.empty(cap, np.uint8)
        self._ck(self._L.pp_debug_prefix(self._h, cap, _ptr(c, _f64p), _ptr(c2, _f64p), _ptr(redone, _u8p)))
        return c[:n_samples], c2[:n_samples], redone[:n_events].astype(bool)

    def debug_lg2_error(self):
        v = _c.c_double()
        self._ck(self._L.pp_debug_lg2_error(self._h, _c.byref(v)))
        return float(v.value)

    def pipeline(self, threshold, rule_mask, duration_gt, duration_lt, min_gt, max_lt, min_width,
                 max_width, window_width, min_gain, filter_ba=None, prefix_mode=PREFIX_AUTO,
                 with_stats=True, host_trace=None, chunk_samples=0, export=False):
        """Whole pipeline on the resident trace, or -- with `host_trace` (float32 or an AdcTrace, ideally pinned) --
        streamed from host memory in chunks that overlap the copy with the computation.  With `export=True`
        the event and segment tables also arrive in page-locked host memory chunk by chunk (keys `event_table`,
        `segment_table` of the result: views of the context's pinned arena, valid until its next pinned use)."""
        p, keep = self._params(threshold, rule_mask, duration_gt, duration_lt, min_gt, max_lt, min_width,
                               max_width, window_width, min_gain, filter_ba, prefix_mode, with_stats)
        out = np.zeros(4, np.int64)
        views = None
        if host_trace is None:
            self._ck(self._L.pp_pipeline(self._h, _c.byref(p), _ptr(out, _i64p)))
        else:
            adc = isinstance(host_trace, AdcTrace)
            x = host_trace.counts if adc else np.ascontiguousarray(host_trace, np.float32)
            t = None
            if export:
                # upper bounds: an event is a run (>= 1 sample each, in practice far fewer); a segment is at least
                # min_width samples unless it is a whole event
                cap_e = int(x.shape[0] // 256 + 4096)
                cap_s = int(x.shape[0] // max(int(min_width), 1) + cap_e)
                spec = [("ev_start", cap_e, np.int64), ("ev_len", cap_e, np.int64), ("event", cap_s, np.int32),
                        ("start", cap_s, np.int64), ("end", cap_s, np.int64)]
                if with_stats:
                    spec += [(k, cap_s, np.float64) for k in ("mean", "std", "min", "max")]
                views = self._arena_views(spec)
                t = HostTables()
                t.cap_events, t.cap_segments = cap_e, cap_s
                t.ev_start, t.ev_len = views["ev_start"].ctypes.data, views["ev_len"].ctypes.data
                t.seg_event, t.seg_start, t.seg_end = (views["event"].ctypes.data, views["start"].ctypes.data,
                                                       views["end"].ctypes.data)
                if with_stats:
                    t.mean, t.std, t.min, t.max = (views[k].ctypes.data for k in ("mean", "std", "min", "max"))
            if adc:
                r = self._L.pp_pipeline_host_adc16(self._h, x.ctypes.data, x.shape[0], host_trace.scale,
                                                   host_trace.offset, int(chunk_samples), _c.byref(p),
                                                   _c.byref(t) if t is not None else None, _ptr(out, _i64p))
            elif export:
                r = self._L.pp_pipeline_host_tables(self._h, _ptr(x, _f32p), x.shape[0], int(chunk_samples),
                                                    _c.byref(p), _c.byref(t), _ptr(out, _i64p))
            else:
                r = self._L.pp_pipeline_host(self._h, _ptr(x, _f32p), x.shape[0], int(chunk_samples),
                                             _c.byref(p), _ptr(out, _i64p))
            if export and r == PP_ERR_CAPACITY and int(out[3]) > 0:
                views = None   # the host tables were too small: the device tables are complete, fetch them
            else:
                self._ck(r)
        del keep
        res = dict(runs=int(out[0]), events=int(out[1]), event_samples=int(out[2]), segments=int(out[3]))
        if export and host_trace is not None:
            if views is None:
                res["event_table"] = self.events(res["events"])
                res["segment_table"] = self.segments(res["segments"], stats=with_stats)
            else:
                ne, ns = res["events"], res["segments"]
                res["event_table"] = (views["ev_start"][:ne], views["ev_len"][:ne])
                res["segment_table"] = {k: views[k][:ns] for k in views if not k.startswith("ev_")}
        return res

    @staticmethod
    def _params(threshold, rule_mask, duration_gt, duration_lt, min_gt, max_lt, min_width, max_width,
                window_width, min_gain, filter_ba=None, prefix_mode=PREFIX_AUTO, with_stats=True):
        p = PipelineParams()
        p.threshold = float(threshold)
        p.rule_mask = int(rule_mask)
        p.duration_gt, p.duration_lt = int(duration_gt), int(duration_lt)
        p.min_gt, p.max_lt = float(min_gt), float(max_lt)
        keep = []
        if filter_ba is not None:
            b, a, zi = [np.ascontiguousarray(v, np.float64) for v in filter_ba]
            keep = [b, a, zi]
            p.filter_ncoef = b.shape[0]
            p.filter_b, p.filter_a, p.filter_zi = _ptr(b, _f64p), _ptr(a, _f64p), _ptr(zi, _f64p)
        else:
            p.filter_ncoef = 0
        p.min_width, p.max_width, p.window_width = int(min_width), int(max_width), int(window_width)
        p.min_gain = float(min_gain)
        p.prefix_mode = int(prefix_mode)
        p.with_stats = int(bool(with_stats))
        return p, keep

    # -- HMM decoding (csrc/hmm.cuh) -----------------------------------------------
    @staticmethod
    def _hmm(model):
        """pp_hmm over the log-space arrays of `model` (a pypore_b200.hmm.HMM); the arrays outlive the call."""
        m = Hmm()
        m.n_states = int(model.n_states)
        for name in ("mean", "inv_std", "log_norm", "log_start", "log_trans"):
            setattr(m, name, _ptr(getattr(model, name), _f64p))
        m.log_end = _ptr(model.log_end, _f64p)
        return m

    def hmm_decode(self, model, algorithm="viterbi", merge=False):
        """Decode the resident segment table, one sequence of segment means per event (pp_hmm_decode); with
        merge=True (Viterbi) runs of segments sharing a state become one segment.  Returns the segment count."""
        n = _i64()
        self._ck(self._L.pp_hmm_decode(self._h, _c.byref(self._hmm(model)), HMM_ALGORITHMS[algorithm],
                                       int(bool(merge)), _c.byref(n)))
        return int(n.value)

    def hmm_decode_sequences(self, model, algorithm, seqs):
        """Decode host sequences (float64 arrays, none empty) in one device call."""
        lens = np.asarray([len(q) for q in seqs], np.int64)
        x = np.ascontiguousarray(np.concatenate(seqs) if len(seqs) else np.zeros(0), np.float64)
        self._ck(self._L.pp_hmm_decode_sequences(self._h, _c.byref(self._hmm(model)), HMM_ALGORITHMS[algorithm],
                                                 _ptr(x, _f64p), _ptr(lens, _i64p), lens.shape[0]))
        return lens

    def hmm_download(self, n_seq, n_states=None):
        """(log-probabilities [n_seq], states [n_states] int32 or None) of the last decode."""
        logp = np.empty(n_seq, np.float64)
        state = np.empty(n_states, np.int32) if n_states is not None else None
        self._ck(self._L.pp_hmm_download(self._h, n_seq, _ptr(logp, _f64p), n_states or 0, _ptr(state, _i32p)))
        return logp, state

    # -- multi-GPU (driven by pypore_b200.dist) ----------------------------------
    def shard_scan(self, threshold, scan_len, dev_record_ptr):
        self._ck(self._L.pp_shard_scan(self._h, float(threshold), int(scan_len), _c.c_void_p(int(dev_record_ptr))))

    def shard_finish(self, threshold, rules, min_width, max_width, window_width, min_gain, skip_first, skip_last,
                     event, dev_record_ptr):
        p, keep = self._params(threshold, min_width=min_width, max_width=max_width, window_width=window_width,
                               min_gain=min_gain, **rules)
        has = event is not None
        self._ck(self._L.pp_shard_finish(self._h, _c.byref(p), int(bool(skip_first)), int(bool(skip_last)),
                                         int(has), int(event[0]) if has else 0, int(event[1]) if has else 0,
                                         _c.c_void_p(int(dev_record_ptr))))

    def shard_plan(self, dev_infos_ptr, rank, world, threshold, rules, halo_avail, dev_plan_ptr):
        """This rank's boundary plan derived on the device from the all-gathered boundary records."""
        p, keep = self._params(threshold, min_width=0, max_width=0, window_width=2, min_gain=0.0, **rules)
        self._ck(self._L.pp_shard_plan(self._h, _c.c_void_p(int(dev_infos_ptr)), int(rank), int(world), _c.byref(p),
                                       int(halo_avail), _c.c_void_p(int(dev_plan_ptr))))

    def shard_finish_planned(self, threshold, rules, min_width, max_width, window_width, min_gain, dev_plan_ptr,
                             dev_record_ptr):
        p, keep = self._params(threshold, min_width=min_width, max_width=max_width, window_width=window_width,
                               min_gain=min_gain, **rules)
        self._ck(self._L.pp_shard_finish_planned(self._h, _c.byref(p), _c.c_void_p(int(dev_plan_ptr)),
                                                 _c.c_void_p(int(dev_record_ptr))))

    def shard_commit(self, rec):
        rec = np.ascontiguousarray(rec, np.int64)
        self._ck(self._L.pp_shard_commit(self._h, _ptr(rec, _i64p)))

    def pack_tables(self, dev_records_ptr, rank, sample_offset, dev_out_ptr, cap_words):
        self._ck(self._L.pp_pack_tables(self._h, _c.c_void_p(int(dev_records_ptr)), int(rank), int(sample_offset),
                                        _c.c_void_p(int(dev_out_ptr)), int(cap_words)))


    # -- control records over peer memory (pp_ctl_*) -----------------------------------------------------------
    def ctl_create(self, rank, world):
        """Allocate this rank's record buffer; returns (64-byte CUDA IPC handle, device pointer)."""
        h = (_c.c_char * 64)()
        p = _c.c_void_p()
        self._ck(self._L.pp_ctl_create(self._h, int(rank), int(world), _c.cast(h, _c.c_void_p), _c.byref(p)))
        return bytes(h), int(p.value)

    def ctl_open(self, handles=None, local_ptrs=None):
        """Map every rank's record buffer: `handles` = the world x 64 bytes of IPC handles (other processes), or
        `local_ptrs` = the device pointers themselves (contexts of this process)."""
        if local_ptrs is not None:
            arr = (_c.c_void_p * len(local_ptrs))(*[_c.c_void_p(int(p)) for p in local_ptrs])
            self._ck(self._L.pp_ctl_open(self._h, None, arr))
        else:
            buf = _c.create_string_buffer(bytes(handles), len(handles))
            self._ck(self._L.pp_ctl_open(self._h, _c.cast(buf, _c.c_void_p), None))

    def ctl_exchange(self, dev_src_ptr, n_words, dev_dst_ptr):
        self._ck(self._L.pp_ctl_exchange(self._h, _c.c_void_p(int(dev_src_ptr)), int(n_words),
                                         _c.c_void_p(int(dev_dst_ptr))))

    def unpack_tables(self, dev_gathered_ptr, world, words_per_rank, dev_records_ptr, n_events, n_segments,
                      stream=None, slot=0, staging_ptr=None, ranks=None):
        """The all-gathered packed tables as host tables, one array per column (views of one of the context's two
        pinned table arenas, valid until that arena's next use): ev_start, ev_len, seg_event, seg_start, seg_end
        [int64], mean, std, min, max [float64].  With `stream` (a cudaStream_t as an integer) the kernel is only
        enqueued there and the caller synchronises before it reads.  With `staging_ptr` (device memory of
        unpacked_bytes() bytes) the kernel writes the same layout THERE and (views, whole arena as bytes) comes
        back: the caller moves it with one device-to-host copy.  `ranks` = (lo, hi): only the rows of those ranks,
        from index 0 (n_events / n_segments are then the counts of that range)."""
        cols_e, cols_i, cols_f = ("ev_start", "ev_len"), ("seg_event", "seg_start", "seg_end"), ("mean", "std", "min", "max")
        spec = ([(k, n_events, np.int64) for k in cols_e] + [(k, n_segments, np.int64) for k in cols_i] +
                [(k, n_segments, np.float64) for k in cols_f])
        total = sum(((n * 8 + 63) // 64) * 64 for _, n, _ in spec) + 64
        arenas = self.__dict__.setdefault("_table_arenas", {})
        arena = arenas.get(slot)
        if arena is None or arena[1] < total:
            if arena is not None:
                self.sync()
                self._L.pp_host_free(self._h, arena[0])
            p = _c.c_void_p()
            cap = int(total * 1.25)
            self._ck(self._L.pp_host_alloc(self._h, cap, _c.byref(p)))
            arenas[slot] = arena = (p.value, cap)
            self._pinned_keep = getattr(self, "_pinned_keep", [])
        v, off = {}, 0
        for name, n, dt in spec:
            buf = (_c.c_char * max(n * 8, 1)).from_address(arena[0] + off)
            v[name] = np.frombuffer(buf, dtype=dt, count=n)
            off += ((n * 8 + 63) // 64) * 64
        t = UnpackedTables()
        t.cap_events, t.cap_segments = int(n_events), int(n_segments)
        for k in cols_e + cols_i + cols_f:
            # staged: same layout in a device arena; the caller copies arena to arena (one DMA transfer)
            setattr(t, k, v[k].ctypes.data if staging_ptr is None else int(staging_ptr) + (v[k].ctypes.data - arena[0]))
        lo, hi = ranks if ranks is not None else (0, int(world))
        self._ck(self._L.pp_unpack_tables_range(self._h, _c.c_void_p(int(dev_gathered_ptr)), int(world),
                                                int(words_per_rank), _c.c_void_p(int(dev_records_ptr)), int(lo), int(hi),
                                                _c.byref(t), 1 if staging_ptr is None else 0,
                                                _c.c_void_p(int(stream)) if stream else None))
        if staging_ptr is not None:
            whole = np.frombuffer((_c.c_char * total).from_address(arena[0]), dtype=np.uint8, count=total)
            return v, whole
        return v

    @staticmethod
    def unpacked_bytes(n_events, n_segments):
        """Size of the arena unpack_tables lays the columns out in."""
        return (2 * (((n_events * 8 + 63) // 64) * 64) + 7 * (((n_segments * 8 + 63) // 64) * 64)) + 64


_default = {}


def default_context(device=None):
    """Process-wide context per device (created on first use)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("PYPORE_B200_USE_LOCAL_RANK") else 0
    ctx = _default.get(device)
    if ctx is None:
        ctx = Context(device)
        _default[device] = ctx
    return ctx
