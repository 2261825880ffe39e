"""Thin object layer over the C-ABI: Context (one per GPU), EventLog (CSR log resident in HBM), detect()."""
import ctypes as C

import numpy as np

from . import _abi
from ._lib import check, lib


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


def _batch(trace_idx, batch_off, act, ts_ms):
    """An appended batch as the C-ABI takes it: (trace_idx int64, batch_off int64, act int32, ts_ms int64)."""
    out = (np.ascontiguousarray(trace_idx, dtype=np.int64), np.ascontiguousarray(batch_off, dtype=np.int64),
           np.ascontiguousarray(act, dtype=np.int32), np.ascontiguousarray(ts_ms, dtype=np.int64))
    if len(out[1]) != len(out[0]) + 1:
        raise ValueError("batch_off must have one entry more than trace_idx")
    if len(out[2]) != len(out[3]):
        raise ValueError("act and ts_ms must have the same length")
    if out[1][-1] != len(out[2]):   # the library copies batch_off[-1] events: it must be exactly the arrays' length
        raise ValueError(f"batch_off[-1] = {int(out[1][-1])} but act / ts_ms hold {len(out[2])} events")
    return out


class Context:
    """siesta_ctx: one per (process, device)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        check(lib().siesta_init(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            lib().siesta_shutdown(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def load_log(self, trace_off, act, ts_ms, n_activities):
        return EventLog(self, trace_off, act, ts_ms, n_activities)

    def wrap_log(self, d_trace_off, d_act, d_ts_ms, n_activities, max_trace_len=0):
        """Borrow torch CUDA tensors (int64, int32, int64) as a resident log."""
        return EventLog(self, None, None, None, n_activities, device_tensors=(d_trace_off, d_act, d_ts_ms),
                        max_trace_len=max_trace_len)

    def evaluate_events(self, trace_off, act, ts_ms, n_activities, nfa, flags=0, copy=True):
        """Literal SaseConnector.evaluate: events travel host -> device inside the call (streamed in chunks).
        An activity column of dtype uint8 (alphabets of at most 256 activities) crosses the link as it is.
        copy=False returns zero-copy views of the library's pinned result block; call .close() on the result."""
        trace_off = np.ascontiguousarray(trace_off, dtype=np.int64)
        ts_ms = np.ascontiguousarray(ts_ms, dtype=np.int64)
        out = C.POINTER(_abi.Matches)()
        if np.asarray(act).dtype == np.uint8:   # byte activity column: siesta_evaluate_events_act8 (1 B/event on the host link)
            act = np.ascontiguousarray(act)
            fn = lib().siesta_evaluate_events_act8
        else:
            act = np.ascontiguousarray(act, dtype=np.int32)
            fn = lib().siesta_evaluate_events
        check(fn(self._h, _ptr(trace_off), _ptr(act), _ptr(ts_ms), len(trace_off) - 1, len(act),
                 n_activities, C.byref(nfa), flags, C.byref(out)))
        if not copy:
            return _abi.MatchResult.from_struct(out.contents, copy=False, free=lambda: lib().siesta_matches_free(out))
        res = _abi.MatchResult.from_struct(out.contents)
        lib().siesta_matches_free(out)
        return res


class EventLog:
    """siesta_log: CSR event log (trace_off int64[T+1], act int32[E], ts_ms int64[E]) in HBM."""

    def __init__(self, ctx, trace_off, act, ts_ms, n_activities, device_tensors=None, max_trace_len=0):
        self.ctx = ctx
        self._h = C.c_void_p()
        self.n_activities = int(n_activities)
        if device_tensors is None:
            trace_off = np.ascontiguousarray(trace_off, dtype=np.int64)
            act = np.ascontiguousarray(act, dtype=np.int32)
            ts_ms = np.ascontiguousarray(ts_ms, dtype=np.int64)
            if len(act) != len(ts_ms):
                raise ValueError("act and ts_ms must have the same length")
            check(lib().siesta_log_load(ctx._h, _ptr(trace_off), _ptr(act), _ptr(ts_ms), len(trace_off) - 1, len(act),
                                        self.n_activities, C.byref(self._h)))
            self._keep = None
        else:
            d_off, d_act, d_ts = device_tensors
            self._keep = device_tensors  # the caller's tensors must outlive the log
            check(lib().siesta_log_wrap_device(ctx._h, C.c_void_p(d_off.data_ptr()), C.c_void_p(d_act.data_ptr()),
                                               C.c_void_p(d_ts.data_ptr()), d_off.numel() - 1, d_act.numel(),
                                               self.n_activities, int(max_trace_len), C.byref(self._h)))
        self.n_traces = lib().siesta_log_n_traces(self._h)
        self.n_events = lib().siesta_log_n_events(self._h)

    @classmethod
    def _adopt(cls, ctx, handle, n_activities):
        """An EventLog over a siesta_log the library created (derived logs)."""
        self = cls.__new__(cls)
        self.ctx, self._h, self.n_activities, self._keep = ctx, handle, int(n_activities), None
        self.n_traces = lib().siesta_log_n_traces(handle)
        self.n_events = lib().siesta_log_n_events(handle)
        return self

    def filter_time(self, from_ms=None, till_ms=None):
        """siesta_log_filter_time: Trace.filter(from, till) on the device -> a new resident EventLog."""
        h = C.c_void_p()
        check(lib().siesta_log_filter_time(self._h, int(from_ms or 0), 0 if from_ms is None else 1, int(till_ms or 0),
                                           0 if till_ms is None else 1, C.byref(h)))
        return EventLog._adopt(self.ctx, h, self.n_activities)

    def group(self, groups, types):
        """siesta_log_group: groups = list of lists of trace indices, types = the query's activity ids ->
        (EventLog whose traces are the kept groups' merged streams, 1-based group ids of those traces)."""
        off = np.zeros(len(groups) + 1, dtype=np.int64)
        np.cumsum([len(g) for g in groups], out=off[1:])
        flat = np.array([t for g in groups for t in g], dtype=np.int64)
        ty = np.asarray(sorted(set(types)), dtype=np.int32)
        gids = np.zeros(max(len(groups), 1), dtype=np.int32)
        h, k = C.c_void_p(), C.c_int32(0)
        check(lib().siesta_log_group(self._h, _ptr(off), _ptr(flat) if len(flat) else None, len(groups), _ptr(ty), len(ty), C.byref(h),
                                     _ptr(gids), C.byref(k)))
        return EventLog._adopt(self.ctx, h, self.n_activities), gids[:k.value].copy()

    def append(self, trace_idx, batch_off, act, ts_ms, n_new_traces=0, n_activities=None):
        """siesta_log_append: a new resident EventLog = this log with the batch appended (events [batch_off[i],
        batch_off[i + 1]) go after the events of trace trace_idx[i]; indices >= n_traces are new traces) ->
        (EventLog, kernel_ms).  This log is not modified and stays usable; close it when no request needs it."""
        ti, bo, a, ts = _batch(trace_idx, batch_off, act, ts_ms)
        n_act = self.n_activities if n_activities is None else int(n_activities)
        h, ms = C.c_void_p(), C.c_double(0.0)
        check(lib().siesta_log_append(self._h, _ptr(ti), _ptr(bo), len(ti), _ptr(a), _ptr(ts), int(n_new_traces), n_act,
                                      C.byref(h), C.byref(ms)))
        return EventLog._adopt(self.ctx, h, n_act), ms.value

    def read(self, t0=0, t1=None):
        """siesta_log_read: host copy of traces [t0, t1) -> (trace_off as stored, act, ts_ms)."""
        t1 = self.n_traces if t1 is None else int(t1)
        off = np.zeros(max(t1 - int(t0), 0) + 1, dtype=np.int64)
        check(lib().siesta_log_read(self._h, int(t0), t1, _ptr(off), None, None))
        n = int(off[-1] - off[0])
        act = np.zeros(max(n, 1), dtype=np.int32)
        ts = np.zeros(max(n, 1), dtype=np.int64)
        check(lib().siesta_log_read(self._h, int(t0), t1, _ptr(off), _ptr(act), _ptr(ts)))
        return off, act[:n], ts[:n]

    def source_events(self):
        """Derived logs: index in the source log of every event."""
        out = np.zeros(max(self.n_events, 1), dtype=np.int64)
        check(lib().siesta_log_source_events(self._h, _ptr(out)))
        return out[:self.n_events]

    def set_first_trace(self, first_trace):
        """This log is the shard starting at global trace `first_trace`: returned trace indices become global."""
        lib().siesta_log_set_first_trace(self._h, int(first_trace))

    def set_blocks(self, local_first, global_first):
        """siesta_log_set_blocks: this log is a block-cyclic shard; block b = local traces [local_first[b], local_first[b + 1])
        = the global traces starting at global_first[b].  Exchange.detect_allgather then overlaps the join with the scan."""
        n = len(global_first)
        assert len(local_first) == n + 1
        lf = (C.c_int64 * (n + 1))(*[int(v) for v in local_first])
        gf = (C.c_int64 * max(n, 1))(*[int(v) for v in global_first])
        check(lib().siesta_log_set_blocks(self._h, n, lf, gf))

    def close(self):
        if self._h:
            lib().siesta_log_free(self._h)
            self._h = C.c_void_p()
            self._keep = None

    def detect(self, nfa, cand=None, flags=0):
        """siesta_detect: host-buffer results (MatchResult)."""
        if cand is not None:
            cand = np.ascontiguousarray(cand, dtype=np.int64)
        out = C.POINTER(_abi.Matches)()
        check(lib().siesta_detect(self._h, C.byref(nfa), _ptr(cand), 0 if cand is None else len(cand), flags, C.byref(out)))
        res = _abi.MatchResult.from_struct(out.contents)
        lib().siesta_matches_free(out)
        return res

    def detect_device(self, nfa, d_cand=None, flags=0, stream=None):
        """siesta_detect_device: results stay in HBM; returns a DeviceMatches (free with .close())."""
        dm = _abi.DevMatches()
        cp = C.c_void_p(d_cand.data_ptr()) if d_cand is not None else None
        n = 0 if d_cand is None else d_cand.numel()
        check(lib().siesta_detect_device(self._h, C.byref(nfa), cp, n, flags, C.c_void_p(stream) if stream else None,
                                         C.byref(dm)))
        return DeviceMatches(dm)

    def detect_device_begin(self, nfa, d_cand=None, flags=0, stream=None):
        """siesta_detect_device_begin: enqueue the verification and return at once; .finish() -> DeviceMatches."""
        h = C.c_void_p()
        cp = C.c_void_p(d_cand.data_ptr()) if d_cand is not None else None
        n = 0 if d_cand is None else d_cand.numel()
        check(lib().siesta_detect_device_begin(self._h, C.byref(nfa), cp, n, flags, C.c_void_p(stream) if stream else None,
                                               C.byref(h)))
        return PendingDetect(h, (nfa, d_cand))

    def declare_counts(self, k_cap=None):
        """siesta_declare_counts: the integer matrices behind /declare (host copy, DeclareCounts)."""
        import numpy as np
        k_cap = int(k_cap if k_cap is not None else 64)
        n = lib().siesta_declare_counts_size(self.n_activities, k_cap)
        out = np.zeros(n, dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_declare_counts(self._h, k_cap, _ptr(out), C.byref(ms)))
        return _abi.DeclareCounts(out, self.n_activities, k_cap, ms.value)

    def declare_counts_device(self, d_out, k_cap, stream=None):
        """siesta_declare_counts_device: packed int64 result into a caller-owned CUDA tensor (for all-reduce)."""
        ms = C.c_double(0.0)
        check(lib().siesta_declare_counts_device(self._h, int(k_cap), C.c_void_p(d_out.data_ptr()),
                                                 C.c_void_p(stream) if stream else None, C.byref(ms)))
        return ms.value

    def declare_counts_refresh(self, old_log, old, trace_idx):
        """siesta_declare_counts_refresh: this log's counts from `old` (DeclareCounts of old_log, or of an earlier
        refresh) after old_log grew into this log by appends that listed trace_idx (their union, ascending) ->
        DeclareCounts equal to self.declare_counts(old.k_cap).  Only the listed traces are counted again."""
        ti, old_packed = _refresh_args(old_log, old, trace_idx)
        out = np.zeros(lib().siesta_declare_counts_size(self.n_activities, old.k_cap), dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_declare_counts_refresh(old_log._h, self._h, _ptr(ti) if len(ti) else None, len(ti), int(old.k_cap),
                                                  _ptr(old_packed), _ptr(out), C.byref(ms)))
        return _abi.DeclareCounts(out, self.n_activities, old.k_cap, ms.value)

    def declare_counts_refresh_device(self, old_log, d_old, d_out, trace_idx, k_cap, stream=None):
        """siesta_declare_counts_refresh_device: d_old (packed counts of old_log, CUDA int64 tensor) -> d_out (this log's
        layout; may be d_old when the alphabet did not grow) -> kernel_ms."""
        ti = np.ascontiguousarray(trace_idx, dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_declare_counts_refresh_device(old_log._h, self._h, _ptr(ti) if len(ti) else None, len(ti), int(k_cap),
                                                         C.c_void_p(d_old.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                                         C.c_void_p(stream) if stream else None, C.byref(ms)))
        return ms.value

    def pair_stats(self, pairs):
        """siesta_pair_stats: the Count record of each (A,B) pair (kernel K4) -> list of dicts with exact python ints."""
        pa = np.array([p[0] for p in pairs], dtype=np.int32)
        pb = np.array([p[1] for p in pairs], dtype=np.int32)
        out = (_abi.PairCount * len(pairs))()
        ms = C.c_double(0.0)
        check(lib().siesta_pair_stats(self._h, _ptr(pa), _ptr(pb), len(pairs), out, C.byref(ms)))
        return [{"count": o.count, "sum": o.sum_duration_ms, "min": o.min_duration_ms, "max": o.max_duration_ms,
                 "sum_squares": o.sum_squares_lo | (o.sum_squares_hi << 64)} for o in out], ms.value

    def pair_stats_device(self, pairs, d_out, stream=None):
        """siesta_pair_stats_device: packed int64[8 * n_pairs] (count, sum, min, max, 4 limbs) into a CUDA tensor."""
        pa = np.array([p[0] for p in pairs], dtype=np.int32)
        pb = np.array([p[1] for p in pairs], dtype=np.int32)
        ms = C.c_double(0.0)
        check(lib().siesta_pair_stats_device(self._h, _ptr(pa), _ptr(pb), len(pairs), C.c_void_p(d_out.data_ptr()),
                                             C.c_void_p(stream) if stream else None, C.byref(ms)))
        return ms.value

    def explore_accurate(self, pattern_activities, candidates, flags=0):
        """siesta_explore_accurate -> (completions int64[n], sum_duration_ms int64[n], kernel_ms)."""
        pa = np.asarray(pattern_activities, dtype=np.int32)
        ca = np.asarray(candidates, dtype=np.int32)
        comp = np.zeros(max(len(ca), 1), dtype=np.int64)
        dur = np.zeros(max(len(ca), 1), dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_explore_accurate(self._h, _ptr(pa), len(pa), _ptr(ca), len(ca), flags, _ptr(comp), _ptr(dur),
                                            C.byref(ms)))
        return comp[:len(ca)], dur[:len(ca)], ms.value

    def why_not_match(self, pattern_activities, constraints, uncertainty, step, k, cand=None, flags=0):
        """siesta_why_not_match (WhyNotMatchSASE.evaluate): constraints = [(pos_a, pos_b, kind, method, value)],
        cand = the traces without a true occurrence (None: every trace) -> _abi.AlmostMatchResult."""
        pa = np.asarray(pattern_activities, dtype=np.int32)
        cons, n_cons = _abi.make_wnm_constraints(constraints)
        out = C.POINTER(_abi.AlmostMatches)()
        n_cand = 0
        if cand is not None:   # an empty list means "no trace", a null pointer "every trace"
            n_cand = len(cand)
            cand = np.ascontiguousarray(cand if n_cand else [0], dtype=np.int64)
        check(lib().siesta_why_not_match(self._h, _ptr(pa), len(pa), C.cast(cons, C.c_void_p), n_cons, int(uncertainty), int(step),
                                         int(k), _ptr(cand), n_cand, flags, C.byref(out)))
        res = _abi.AlmostMatchResult(out.contents)
        lib().siesta_almost_matches_free(out)
        return res

    def build_index(self, pairs):
        """siesta_index_build: posting lists of the (A,B) pairs from the resident log (SeqTable view)."""
        return PairIndex(self, pairs)

    def load_index(self, pairs, lists):
        """siesta_index_load: posting lists (ascending trace indices) produced elsewhere, e.g. index.parquet."""
        return PairIndex(self, pairs, lists=lists)


def _refresh_args(old_log, old, trace_idx):
    """(trace_idx int64, old packed counts) of a count refresh; the counts must be laid out for old_log's alphabet."""
    if old.n_activities != old_log.n_activities:
        raise ValueError(f"the old counts are for {old.n_activities} activities, old_log has {old_log.n_activities}")
    return np.ascontiguousarray(trace_idx, dtype=np.int64), np.ascontiguousarray(old.packed, dtype=np.int64)


def _flat_lists(lists):
    """Posting lists back to back as the C-ABI takes them: (offsets int64[n + 1], entries int64)."""
    lists = [np.ascontiguousarray(x, dtype=np.int64) for x in lists]
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=off[1:])
    flat = np.concatenate(lists) if lists and off[-1] else np.zeros(0, dtype=np.int64)
    return off, flat


class PairIndex:
    """siesta_index: per-pair posting lists in HBM + the sorted trace-id intersection (kernel K2)."""

    def __init__(self, log, pairs, lists=None):
        self.log = log
        self.pairs = [(int(a), int(b)) for a, b in pairs]
        pa = np.array([p[0] for p in self.pairs], dtype=np.int32)
        pb = np.array([p[1] for p in self.pairs], dtype=np.int32)
        self._h = C.c_void_p()
        if lists is None:
            check(lib().siesta_index_build(log._h, _ptr(pa), _ptr(pb), len(self.pairs), C.byref(self._h)))
        else:
            off, flat = _flat_lists(lists)
            check(lib().siesta_index_load(log._h, len(self.pairs), _ptr(pa), _ptr(pb), _ptr(off), _ptr(flat), C.byref(self._h)))

    def _adopt(self, new_log, h):
        out = PairIndex.__new__(PairIndex)
        out.log, out.pairs, out._h = new_log, list(self.pairs), h
        return out

    def append(self, new_log, lists):
        """siesta_index_append: a new index on new_log (this log with batches appended) whose list p = this list p UNION
        lists[p] (ascending trace indices of new_log, aligned with self.pairs; an empty array leaves the pair as it is),
        e.g. a batch's index.parquet rows read by ingest.read_index_table -> (PairIndex, kernel_ms).  This index is not
        modified and stays usable; the result counts as loaded lists."""
        if len(lists) != len(self.pairs):
            raise ValueError(f"{len(lists)} delta lists for an index of {len(self.pairs)} pairs")
        off, flat = _flat_lists(lists)
        h, ms = C.c_void_p(), C.c_double(0.0)
        check(lib().siesta_index_append(self._h, new_log._h, _ptr(off), _ptr(flat), C.byref(h), C.byref(ms)))
        return self._adopt(new_log, h), ms.value

    def refresh(self, new_log, trace_idx):
        """siesta_index_refresh (built indexes only): re-derive the traces a log append listed (trace_idx as passed to
        EventLog.append) on new_log and merge -> (PairIndex equal to new_log.build_index(self.pairs), kernel_ms).  This
        index is not modified and stays usable."""
        ti = np.ascontiguousarray(trace_idx, dtype=np.int64)
        h, ms = C.c_void_p(), C.c_double(0.0)
        check(lib().siesta_index_refresh(self._h, new_log._h, _ptr(ti) if len(ti) else None, len(ti), C.byref(h), C.byref(ms)))
        return self._adopt(new_log, h), ms.value

    def close(self):
        if self._h:
            lib().siesta_index_free(self._h)
            self._h = C.c_void_p()

    def posting_list(self, i):
        n = lib().siesta_index_list_len(self._h, i)
        out = np.zeros(max(n, 0), dtype=np.int64)
        check(lib().siesta_index_get_list(self._h, i, _ptr(out), len(out)))
        return out

    def intersect(self, pair_ids=None):
        """getCommonIds: ascending trace indices present in every selected posting list."""
        ids = np.arange(len(self.pairs), dtype=np.int32) if pair_ids is None else np.asarray(pair_ids, dtype=np.int32)
        cap = min(lib().siesta_index_list_len(self._h, int(i)) for i in ids) if len(ids) else 0
        out = np.zeros(max(cap, 0), dtype=np.int64)
        n = C.c_int64(0)
        check(lib().siesta_intersect(self._h, _ptr(ids), len(ids), _ptr(out), len(out), C.byref(n)))
        return out[:n.value].copy()

    def intersect_device_ms(self, pair_ids=None):
        """siesta_intersect_device with the result left (and freed) in HBM -> (n_common, kernel_ms): the device-side cost."""
        ids = np.arange(len(self.pairs), dtype=np.int32) if pair_ids is None else np.asarray(pair_ids, dtype=np.int32)
        d_out, n, ms = C.c_void_p(), C.c_int64(0), C.c_double(0.0)
        check(lib().siesta_intersect_device(self._h, _ptr(ids), len(ids), C.byref(d_out), C.byref(n), C.byref(ms)))
        lib().siesta_device_free(self.log._h, d_out)
        return n.value, ms.value

    def candidates(self, expansions):
        """siesta_candidates: union over the expansions (lists of pair ids) of the intersection of their posting lists."""
        off = np.zeros(len(expansions) + 1, dtype=np.int32)
        np.cumsum([len(x) for x in expansions], out=off[1:])
        ids = np.array([i for x in expansions for i in x], dtype=np.int32)
        out = np.zeros(max(self.log.n_traces, 1), dtype=np.int64)
        n = C.c_int64(0)
        check(lib().siesta_candidates(self._h, _ptr(off), _ptr(ids), len(expansions), _ptr(out), len(out), C.byref(n)))
        return out[:n.value].copy()


class Exchange:
    """siesta_exchange: this rank's end of the device-side joins (csrc/multi.cu).  Create one per rank with the same
    world / capacity, connect the peers (export() / import_peer() across processes, connect_local() inside one), then
    call the collectives in the same order on every rank."""

    def __init__(self, ctx, world, rank, capacity_bytes):
        self.ctx, self.world, self.rank, self.capacity = ctx, int(world), int(rank), int(capacity_bytes)
        self._h = C.c_void_p()
        check(lib().siesta_exchange_create(ctx._h, self.world, self.rank, self.capacity, C.byref(self._h)))

    def export(self):
        buf = (C.c_ubyte * _abi.EXCHANGE_HANDLE_BYTES)()
        check(lib().siesta_exchange_export(self._h, buf))
        return bytes(buf)

    def import_peer(self, peer_rank, handle):
        buf = (C.c_ubyte * _abi.EXCHANGE_HANDLE_BYTES).from_buffer_copy(handle)
        check(lib().siesta_exchange_import(self._h, int(peer_rank), buf))

    def connect_local(self, peer):
        check(lib().siesta_exchange_connect_local(self._h, peer.rank, peer._h))

    def detect_allgather(self, log, nfa, flags=0):
        """siesta_detect_allgather -> (DeviceMatches of ALL ranks, ExchangeStats)."""
        dm, st = _abi.DevMatches(), _abi.ExchangeStats()
        check(lib().siesta_detect_allgather(log._h, C.byref(nfa), flags, self._h, C.byref(dm), C.byref(st)))
        return DeviceMatches(dm), st

    def allreduce_i64(self, d_buf, op=_abi.REDUCE_SUM, stream=None):
        """In-place all-reduce of an int64 CUDA tensor over the peer regions."""
        check(lib().siesta_exchange_allreduce_i64(self._h, C.c_void_p(d_buf.data_ptr()), d_buf.numel(), int(op),
                                                  C.c_void_p(stream) if stream else None))
        return d_buf

    def close(self):
        if self._h:
            lib().siesta_exchange_free(self._h)
            self._h = C.c_void_p()


class Multi:
    """siesta_multi: ONE process driving several GPUs (what a single JVM does).  device_ids may repeat a device."""

    def __init__(self, device_ids):
        ids = np.asarray(device_ids, dtype=np.int32)
        self._h = C.c_void_p()
        check(lib().siesta_multi_init(_ptr(ids), len(ids), C.byref(self._h)))
        self.n_devices = len(ids)

    def load_log(self, trace_off, act, ts_ms, n_activities):
        return MultiLog(self, trace_off, act, ts_ms, n_activities)

    def close(self):
        if self._h:
            lib().siesta_multi_shutdown(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class MultiLog:
    """siesta_multi_log: a host CSR log sharded over the devices of a Multi by contiguous trace range."""

    def __init__(self, multi, trace_off, act, ts_ms, n_activities):
        trace_off = np.ascontiguousarray(trace_off, dtype=np.int64)
        act = np.ascontiguousarray(act, dtype=np.int32)
        ts_ms = np.ascontiguousarray(ts_ms, dtype=np.int64)
        self.multi, self.n_activities = multi, int(n_activities)
        self._h = C.c_void_p()
        check(lib().siesta_multi_log_load(multi._h, _ptr(trace_off), _ptr(act), _ptr(ts_ms), len(trace_off) - 1, len(act),
                                          self.n_activities, C.byref(self._h)))

    def append(self, trace_idx, batch_off, act, ts_ms, n_new_traces=0, n_activities=None):
        """siesta_multi_log_append: EventLog.append with GLOBAL trace indices; new traces go to the last shard ->
        a new MultiLog (this one is not modified)."""
        ti, bo, a, ts = _batch(trace_idx, batch_off, act, ts_ms)
        n_act = self.n_activities if n_activities is None else int(n_activities)
        h = C.c_void_p()
        check(lib().siesta_multi_log_append(self._h, _ptr(ti), _ptr(bo), len(ti), _ptr(a), _ptr(ts), int(n_new_traces), n_act,
                                            C.byref(h)))
        new = MultiLog.__new__(MultiLog)
        new.multi, new.n_activities, new._h = self.multi, n_act, h
        return new

    def detect(self, nfa, flags=0):
        out = C.POINTER(_abi.Matches)()
        check(lib().siesta_multi_detect(self._h, C.byref(nfa), flags, C.byref(out)))
        res = _abi.MatchResult.from_struct(out.contents)
        lib().siesta_matches_free(out)
        return res

    def why_not_match(self, pattern_activities, constraints, uncertainty, step, k, cand=None, flags=0):
        """siesta_multi_why_not_match: cand = ascending GLOBAL trace indices (None: every trace)."""
        pa = np.asarray(pattern_activities, dtype=np.int32)
        cons, n_cons = _abi.make_wnm_constraints(constraints)
        out = C.POINTER(_abi.AlmostMatches)()
        n_cand = 0
        if cand is not None:
            n_cand = len(cand)
            cand = np.ascontiguousarray(cand if n_cand else [0], dtype=np.int64)
        check(lib().siesta_multi_why_not_match(self._h, _ptr(pa), len(pa), C.cast(cons, C.c_void_p), n_cons, int(uncertainty), int(step),
                                               int(k), _ptr(cand), n_cand, flags, C.byref(out)))
        res = _abi.AlmostMatchResult(out.contents)
        lib().siesta_almost_matches_free(out)
        return res

    def declare_counts(self, k_cap=64):
        n = lib().siesta_declare_counts_size(self.n_activities, int(k_cap))
        out = np.zeros(n, dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_multi_declare_counts(self._h, int(k_cap), _ptr(out), C.byref(ms)))
        return _abi.DeclareCounts(out, self.n_activities, int(k_cap), ms.value)

    def declare_counts_refresh(self, old_log, old, trace_idx):
        """siesta_multi_declare_counts_refresh: EventLog.declare_counts_refresh with GLOBAL trace indices, for this log
        grown from old_log by MultiLog.append."""
        ti, old_packed = _refresh_args(old_log, old, trace_idx)
        out = np.zeros(lib().siesta_declare_counts_size(self.n_activities, old.k_cap), dtype=np.int64)
        ms = C.c_double(0.0)
        check(lib().siesta_multi_declare_counts_refresh(old_log._h, self._h, _ptr(ti) if len(ti) else None, len(ti), int(old.k_cap),
                                                        _ptr(old_packed), _ptr(out), C.byref(ms)))
        return _abi.DeclareCounts(out, self.n_activities, old.k_cap, ms.value)

    def close(self):
        if self._h:
            lib().siesta_multi_log_free(self._h)
            self._h = C.c_void_p()


def exchange_required_bytes(log, nfa, flags=0):
    return int(lib().siesta_exchange_required_bytes(log._h, C.byref(nfa), flags))


class PendingDetect:
    """A verification request whose kernels are enqueued (siesta_detect_device_begin); finish() exactly once."""

    def __init__(self, h, keep):
        self._h, self._keep = h, keep   # nfa / candidates stay alive until finish()

    def finish(self):
        dm = _abi.DevMatches()
        h, self._h = self._h, None
        if h is None:
            raise RuntimeError("PendingDetect.finish() called twice")
        check(lib().siesta_detect_device_finish(h, C.byref(dm)))
        self._keep = None
        return DeviceMatches(dm)


class DeviceMatches:
    def __init__(self, dm):
        self.dm = dm
        for k in ("n_traces", "n_occurrences", "n_events", "n_matches_emitted", "n_ref_errors", "kernel_ms", "detect_ms", "n_unsupported"):
            setattr(self, k, getattr(dm, k))

    def close(self):
        if self.dm is not None:
            lib().siesta_dev_matches_free(C.byref(self.dm))
            self.dm = None

    def tensors(self, device_index=0):
        """Zero-copy torch views of the device result (valid until close()); keys as in MatchResult."""
        import torch

        class _View:
            def __init__(self, ptr, n, typestr):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}

        def view(ptr, n, typestr, dtype):
            if not ptr or n == 0:
                return torch.zeros(0, dtype=dtype, device=f"cuda:{device_index}")
            return torch.as_tensor(_View(ptr, n, typestr), device=f"cuda:{device_index}")

        d = self.dm
        out = {"trace_idx": view(d.d_trace_idx, d.n_traces, "<i8", torch.int64),
               "occ_off": view(d.d_occ_off, d.n_traces + 1, "<i8", torch.int64),
               "ev_off": view(d.d_ev_off, d.n_occurrences + 1, "<i8", torch.int64),
               "ev_pos": view(d.d_ev_pos, d.n_events, "<i4", torch.int32),
               "err_trace_idx": view(d.d_err_trace_idx, d.n_ref_errors, "<i8", torch.int64),
               "unsupported_trace_idx": view(d.d_unsupported_trace_idx, d.n_unsupported, "<i8", torch.int64)}
        if d.d_ev_rank:
            out["ev_rank"] = view(d.d_ev_rank, d.n_events, "<i4", torch.int32)
            out["ev_act"] = view(d.d_ev_act, d.n_events, "<i4", torch.int32)
            out["ev_ts_ms"] = view(d.d_ev_ts_ms, d.n_events, "<i8", torch.int64)
        return out


def kernel_launches():
    return int(lib().siesta_kernel_launches())
