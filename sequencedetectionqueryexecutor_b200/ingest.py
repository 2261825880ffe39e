"""SIESTA bucket tables -> the resident layout of the GPU path (SURVEY.md §8(f) row 1, Appendix C).

The reference reads the tables its preprocess component wrote with Spark:
  seq.parquet / single.parquet  {trace_id: string, event_type: string, timestamp: string "yyyy-MM-dd HH:mm:ss[.f]",
                                 position: int}          S3Connector.querySequenceTableDeclare :299-314, getFromSingle :214-232
  index.parquet                 {eventA, eventB, trace_id: string, positionA, positionB: int   (meta.mode = positions)
                                                                or timestampA, timestampB: timestamp (meta.mode = timestamps)}
                                                                                   S3Connector.getAllEventPairs :236-292
and keeps them as maps of boxed objects.  Here they become the CSR event log (trace offsets, int32 activity ids, int64
epoch milliseconds) and ascending posting lists of dense trace indices, plus the two host dictionaries (activity
names, folded case-insensitively because the engine compares event types with equalsIgnoreCase; trace-id strings).

Host code (pyarrow + numpy, vectorised; no GPU involved): `EventLog` / `PairIndex` of api.py take the arrays as they
are (`Context.load_log`, `EventLog.load_index`).  The writers produce tables of the same schema from a CSR log - used by
the tests and to build synthetic buckets.
"""
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .sase import ActivityDictionary


@dataclass
class SeqLog:
    """A whole log in the GPU path's layout + its dictionaries."""
    trace_off: np.ndarray          # int64 [T + 1]
    act: np.ndarray                # int32 [E] dense activity id
    ts_ms: np.ndarray              # int64 [E] epoch milliseconds
    trace_ids: List[str]           # dense trace index -> trace id
    activities: ActivityDictionary

    @property
    def n_traces(self):
        return len(self.trace_off) - 1

    def trace_index(self):
        """trace id -> dense index"""
        return {t: i for i, t in enumerate(self.trace_ids)}


def _table(src, columns=None):
    import pyarrow as pa
    import pyarrow.parquet as pq
    if isinstance(src, pa.Table):
        return src.select(columns) if columns else src
    return pq.read_table(src, columns=columns)


def timestamps_to_ms(col, tz_offset_ms=0):
    """Column of `yyyy-MM-dd HH:mm:ss[.fffffffff]` strings (what java.sql.Timestamp.valueOf parses, S3Connector.java:307)
    or of arrow timestamps -> int64 epoch milliseconds.  Timestamp.valueOf reads the string in the JVM's default time
    zone; `tz_offset_ms` is that zone's offset (0 = UTC).  Fractions beyond milliseconds are truncated, as
    Timestamp.getTime() does."""
    import pyarrow as pa
    import pyarrow.compute as pc
    if isinstance(col, pa.ChunkedArray):
        col = col.combine_chunks()
    if pa.types.is_timestamp(col.type):
        return np.asarray(pc.cast(col, pa.timestamp("ms"), safe=False).cast(pa.int64()), dtype=np.int64) - tz_offset_ms
    # arrow's string -> timestamp parser accepts the blank between date and time and an optional fraction
    ns = pc.cast(col, pa.timestamp("ns"))
    return np.asarray(pc.cast(ns, pa.timestamp("ms"), safe=False).cast(pa.int64()), dtype=np.int64) - tz_offset_ms


def read_seq_table(src, activities: Optional[ActivityDictionary] = None, tz_offset_ms=0) -> SeqLog:
    """seq.parquet (or single.parquet) -> SeqLog.  Traces are numbered in order of first appearance of their id; the
    events of a trace are ordered by `position` (the order the preprocess wrote; Trace keeps the list "in the correct
    order", J/model/DBModel/Trace.java:14-17), ties by their order in the table."""
    tb = _table(src, ["trace_id", "event_type", "timestamp", "position"])
    n = tb.num_rows
    acts = activities if activities is not None else ActivityDictionary()
    if n == 0:
        return SeqLog(np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int64), [], acts)
    tid_dict = tb["trace_id"].combine_chunks().dictionary_encode()
    ev_dict = tb["event_type"].combine_chunks().dictionary_encode()
    tid_codes = np.asarray(tid_dict.indices, dtype=np.int64)          # dictionary order = first appearance
    trace_ids = [str(x) for x in tid_dict.dictionary.to_pylist()]
    name_to_id = np.array([acts.add(str(x)) for x in ev_dict.dictionary.to_pylist()], dtype=np.int32)  # case-folded
    act = name_to_id[np.asarray(ev_dict.indices, dtype=np.int64)]
    ts = timestamps_to_ms(tb["timestamp"], tz_offset_ms)
    pos = np.asarray(tb["position"].combine_chunks().to_numpy(zero_copy_only=False), dtype=np.int64)
    order = np.lexsort((np.arange(n), pos, tid_codes))                # by trace, then position, then table order
    counts = np.bincount(tid_codes, minlength=len(trace_ids))
    trace_off = np.zeros(len(trace_ids) + 1, dtype=np.int64)
    np.cumsum(counts, out=trace_off[1:])
    return SeqLog(trace_off, np.ascontiguousarray(act[order]), np.ascontiguousarray(ts[order]), trace_ids, acts)


@dataclass
class SeqDelta:
    """A batch of events to append to a resident log (EventLog.append / MultiLog.append take its fields): the events of
    listed trace i are act / ts_ms[batch_off[i]:batch_off[i + 1]] and go after the existing events of trace
    trace_idx[i] (ascending); indices >= the log's trace count are new traces."""
    trace_idx: np.ndarray          # int64 [k] ascending dense trace indices
    batch_off: np.ndarray          # int64 [k + 1]
    act: np.ndarray                # int32 [batch_off[k]]
    ts_ms: np.ndarray              # int64 [batch_off[k]]
    n_new_traces: int
    n_activities: int              # size of the (grown) activity dictionary


def read_seq_delta(src, trace_ids: List[str], activities: ActivityDictionary, trace_lens=None, tz_offset_ms=0) -> SeqDelta:
    """A seq.parquet batch the preprocess wrote after the log became resident -> SeqDelta.  Known trace ids map to their
    dense index; unknown ones are numbered T, T + 1, ... in order of first appearance and appended to `trace_ids`.
    Names go through the same case-folding `activities`, which grows.  Events are ordered by `position`, ties by table
    order (as read_seq_table).  With `trace_lens` (current event count of every known trace), a row whose position lies
    below its trace's length raises ValueError: such a batch rewrites existing events, which an append cannot."""
    tb = _table(src, ["trace_id", "event_type", "timestamp", "position"])
    n, T = tb.num_rows, len(trace_ids)
    if n == 0:
        return SeqDelta(np.zeros(0, dtype=np.int64), np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int32),
                        np.zeros(0, dtype=np.int64), 0, len(activities))
    index_of = {t: i for i, t in enumerate(trace_ids)}
    tid_dict = tb["trace_id"].combine_chunks().dictionary_encode()
    n_new = 0
    dense = []
    for x in tid_dict.dictionary.to_pylist():                         # dictionary order = first appearance
        x = str(x)
        if x not in index_of:
            index_of[x] = T + n_new
            trace_ids.append(x)
            n_new += 1
        dense.append(index_of[x])
    tr = np.asarray(dense, dtype=np.int64)[np.asarray(tid_dict.indices, dtype=np.int64)]
    ev_dict = tb["event_type"].combine_chunks().dictionary_encode()
    name_to_id = np.array([activities.add(str(x)) for x in ev_dict.dictionary.to_pylist()], dtype=np.int32)
    act = name_to_id[np.asarray(ev_dict.indices, dtype=np.int64)]
    ts = timestamps_to_ms(tb["timestamp"], tz_offset_ms)
    pos = np.asarray(tb["position"].combine_chunks().to_numpy(zero_copy_only=False), dtype=np.int64)
    if trace_lens is not None and T:
        lens = np.asarray(trace_lens, dtype=np.int64)
        known = tr < T
        bad = np.zeros(n, dtype=bool)
        bad[known] = pos[known] < lens[tr[known]]
        if bad.any():
            r = int(np.flatnonzero(bad)[0])
            raise ValueError(f"batch row {r} rewrites position {int(pos[r])} of trace {trace_ids[int(tr[r])]!r}, "
                             f"which already holds {int(lens[tr[r]])} events: not an append")
    order = np.lexsort((np.arange(n), pos, tr))                      # by trace, then position, then table order
    trace_idx, counts = np.unique(tr, return_counts=True)
    batch_off = np.zeros(len(trace_idx) + 1, dtype=np.int64)
    np.cumsum(counts, out=batch_off[1:])
    return SeqDelta(trace_idx.astype(np.int64), batch_off, np.ascontiguousarray(act[order]), np.ascontiguousarray(ts[order]),
                    n_new, len(activities))


def merge_delta(trace_off, act, ts_ms, delta: SeqDelta):
    """The append restated on the host: (trace_off, act, ts_ms) of the log with `delta` appended - what
    siesta_log_append builds on the device, and the host copy a caller that keeps one maintains."""
    trace_off = np.asarray(trace_off, dtype=np.int64)
    T = len(trace_off) - 1
    T2 = T + int(delta.n_new_traces)
    old_len = np.zeros(T2, dtype=np.int64)
    old_len[:T] = np.diff(trace_off)
    add = np.zeros(T2, dtype=np.int64)
    add[delta.trace_idx] = np.diff(delta.batch_off)
    new_off = np.zeros(T2 + 1, dtype=np.int64)
    np.cumsum(old_len + add, out=new_off[1:])
    E2 = int(new_off[-1])
    # destination of every old event (shifted by the batch events of earlier traces) and of every batch event
    before = np.zeros(T2 + 1, dtype=np.int64)
    np.cumsum(add, out=before[1:])
    old_trace = np.repeat(np.arange(T), old_len[:T])
    old_dst = np.arange(int(trace_off[-1]), dtype=np.int64) + before[old_trace]
    b_trace = np.repeat(delta.trace_idx, np.diff(delta.batch_off))
    b_rank = np.arange(int(delta.batch_off[-1]), dtype=np.int64) - np.repeat(delta.batch_off[:-1], np.diff(delta.batch_off))
    b_dst = new_off[b_trace] + old_len[b_trace] + b_rank
    out_act = np.zeros(E2, dtype=np.int32)
    out_ts = np.zeros(E2, dtype=np.int64)
    out_act[old_dst] = act
    out_ts[old_dst] = ts_ms
    out_act[b_dst] = delta.act
    out_ts[b_dst] = delta.ts_ms
    return new_off, out_act, out_ts


def read_index_table(src, log: SeqLog, pairs: Optional[Sequence[Tuple[str, str]]] = None):
    """index.parquet -> (pairs [(activity id A, activity id B)], posting lists [ascending int64 dense trace indices]),
    ready for EventLog.load_index.  `pairs` (names) restricts the read to the requested pairs, as getAllEventPairs'
    where-clause does; a trace listed several times under a pair (one row per occurrence pair) appears once (the
    `distinct` of SparkDatabaseRepository.getCommonIds :160-178).  Rows of traces or activities the log does not know
    are dropped."""
    tb = _table(src, ["eventA", "eventB", "trace_id"])
    if tb.num_rows == 0:
        return [], []
    index_of = log.trace_index()
    a_dict = tb["eventA"].combine_chunks().dictionary_encode()
    b_dict = tb["eventB"].combine_chunks().dictionary_encode()
    t_dict = tb["trace_id"].combine_chunks().dictionary_encode()
    a_ids = np.array([log.activities.id(str(x)) for x in a_dict.dictionary.to_pylist()], dtype=np.int64)
    b_ids = np.array([log.activities.id(str(x)) for x in b_dict.dictionary.to_pylist()], dtype=np.int64)
    t_ids = np.array([index_of.get(str(x), -1) for x in t_dict.dictionary.to_pylist()], dtype=np.int64)
    a = a_ids[np.asarray(a_dict.indices, dtype=np.int64)]
    b = b_ids[np.asarray(b_dict.indices, dtype=np.int64)]
    t = t_ids[np.asarray(t_dict.indices, dtype=np.int64)]
    keep = (a >= 0) & (b >= 0) & (t >= 0)
    if pairs is not None:
        want = {(log.activities.id(x), log.activities.id(y)) for x, y in pairs}
        n_act = max(len(log.activities), 1)
        want_keys = np.array(sorted(p[0] * n_act + p[1] for p in want if p[0] >= 0 and p[1] >= 0), dtype=np.int64)
        keep &= np.isin(a * n_act + b, want_keys)
    a, b, t = a[keep], b[keep], t[keep]
    n_act = max(len(log.activities), 1)
    T = max(log.n_traces, 1)
    key = np.unique((a * n_act + b) * T + t)          # sorted: by pair, then trace index; duplicates removed
    pair_key = key // T
    out_pairs, lists = [], []
    if len(key):
        starts = np.flatnonzero(np.concatenate(([True], pair_key[1:] != pair_key[:-1])))
        ends = np.concatenate((starts[1:], [len(key)]))
        for s, e in zip(starts, ends):
            out_pairs.append((int(pair_key[s] // n_act), int(pair_key[s] % n_act)))
            lists.append(np.ascontiguousarray(key[s:e] % T))
    return out_pairs, lists


@dataclass
class Count:
    """A CountTable record (J/model/DBModel/Count.java:12-24)."""
    eventA: str
    eventB: str
    sum_duration: int
    count: int
    min_duration: int
    max_duration: int
    sum_squares: float


def consecutive_pairs(pattern_names: Sequence[str]):
    """SIESTAPattern.extractPairsConsecutive (J/model/Patterns/SIESTAPattern.java:96-105): the pairs (e_i, e_i+1) of the
    pattern's events as a set.  The reference iterates a HashSet (order unspecified); here: pattern order."""
    out = []
    for a, b in zip(pattern_names[:-1], pattern_names[1:]):
        if (a, b) not in out:
            out.append((a, b))
    return out


def read_count_table(src, pairs: Sequence[Tuple[str, str]]) -> List[Count]:
    """/stats as the reference answers it: a lookup in count.parquet (QueryPlanStats.execute, J/model/Queries/QueryPlans/
    QueryPlanStats.java:43-48 -> S3Connector.getCounts :125-169).  A row holds `eventA` and an array of records
    (eventB, sum_duration: long, count: int, min_duration: long, max_duration: long, sum_squares: double), read by
    POSITION as the reference does (row.getSeq(0) / getString(1); struct fields 0..5).  Returns, for every requested pair
    in the requested order, the FIRST stored record of that pair; pairs the table does not hold are skipped (getCounts'
    final loop).  Names compare exactly (String.equals), not case-folded."""
    import pyarrow as pa
    tb = _table(src)
    list_col = next(i for i, f in enumerate(tb.schema) if pa.types.is_list(f.type) or pa.types.is_large_list(f.type))
    name_col = next(i for i, f in enumerate(tb.schema) if pa.types.is_string(f.type) or pa.types.is_large_string(f.type))
    wanted_a = {a for a, _ in pairs}
    found = {}
    names = tb.column(name_col).to_pylist()
    records = tb.column(list_col)
    for r, event_a in enumerate(names):
        if event_a not in wanted_a:          # the where-clause on eventA
            continue
        for rec in records[r].as_py() or []:
            v = list(rec.values()) if isinstance(rec, dict) else list(rec)
            key = (event_a, v[0])
            if key not in found:
                found[key] = Count(event_a, v[0], int(v[1]), int(v[2]), int(v[3]), int(v[4]), float(v[5]))
    return [found[p] for p in pairs if p in found]


def count_table_from_stats(stats: Sequence[Count]):
    """count.parquet rows (pyarrow Table, column order of the preprocess: the record array first, eventA second) of the
    given records - synthetic buckets and tests; the records themselves come from siesta_pair_stats (kernel K4) or from
    the preprocess."""
    import pyarrow as pa
    by_a = {}
    for c in stats:
        by_a.setdefault(c.eventA, []).append({"eventB": c.eventB, "sum_duration": int(c.sum_duration), "count": int(c.count),
                                              "min_duration": int(c.min_duration), "max_duration": int(c.max_duration),
                                              "sum_squares": float(c.sum_squares)})
    rec_t = pa.struct([("eventB", pa.string()), ("sum_duration", pa.int64()), ("count", pa.int32()),
                       ("min_duration", pa.int64()), ("max_duration", pa.int64()), ("sum_squares", pa.float64())])
    return pa.table({"times": pa.array(list(by_a.values()), type=pa.list_(rec_t)),
                     "eventA": pa.array(list(by_a.keys()), type=pa.string())})


def filter_time_range(trace_off, act, ts_ms, from_ms=None, till_ms=None):
    """Trace.filter(from, till) (J/model/DBModel/Trace.java:25-29) for a whole CSR log: keeps the events with
    from <= timestamp <= till (either bound may be None) -> (trace_off, act, ts_ms, kept) where `kept` are the indices of
    the surviving events in the input (in-trace positions of the filtered log are ranks among the kept events, as in the
    reference, which filters the list before Utils.transformToSaseEvents numbers it)."""
    ts_ms = np.asarray(ts_ms, dtype=np.int64)
    keep = np.ones(len(ts_ms), dtype=bool)
    if from_ms is not None:
        keep &= ts_ms >= from_ms
    if till_ms is not None:
        keep &= ts_ms <= till_ms
    csum = np.concatenate(([0], np.cumsum(keep, dtype=np.int64)))
    new_off = csum[np.asarray(trace_off, dtype=np.int64)]
    kept = np.flatnonzero(keep)
    return new_off, np.ascontiguousarray(np.asarray(act)[kept]), np.ascontiguousarray(ts_ms[kept]), kept


# ------------------------------------------------------------------------------------------------ writers (tests, tooling)
def _format_ts(ts_ms):
    base = ts_ms.astype("datetime64[ms]")
    return np.char.replace(np.datetime_as_string(base, unit="ms"), "T", " ")


def seq_table_from_csr(trace_off, act, ts_ms, trace_ids: Sequence[str], activity_names: Sequence[str]):
    """The seq.parquet rows of a CSR log (pyarrow Table; write with pyarrow.parquet.write_table)."""
    import pyarrow as pa
    lens = np.diff(trace_off)
    trace_of = np.repeat(np.arange(len(lens)), lens)
    pos = np.arange(len(act)) - np.repeat(trace_off[:-1], lens)
    names = np.asarray(activity_names, dtype=object)
    tids = np.asarray(trace_ids, dtype=object)
    return pa.table({"trace_id": pa.array(tids[trace_of], type=pa.string()),
                     "event_type": pa.array(names[act], type=pa.string()),
                     "timestamp": pa.array(_format_ts(np.asarray(ts_ms, dtype=np.int64)), type=pa.string()),
                     "position": pa.array(pos.astype(np.int32), type=pa.int32())})


def index_table_from_csr(trace_off, act, trace_ids: Sequence[str], activity_names: Sequence[str], pairs):
    """index.parquet rows (meta.mode = positions) of the given (A, B) activity-id pairs under the SeqTable view: for every
    trace that holds an A before a B, ONE row with the first A and the last B (for A == B: the first two occurrences).
    The preprocess writes one row per extracted occurrence pair under its own policy (not in the reference repository);
    posting-list membership - all that the pruning step reads - is the same."""
    import pyarrow as pa
    rows = {"eventA": [], "eventB": [], "trace_id": [], "positionA": [], "positionB": []}
    for t in range(len(trace_off) - 1):
        seg = act[trace_off[t]:trace_off[t + 1]]
        for a, b in pairs:
            ia = np.flatnonzero(seg == a)
            ib = np.flatnonzero(seg == b)
            if a == b:
                if len(ia) >= 2:
                    pa_, pb_ = ia[0], ia[1]
                else:
                    continue
            elif len(ia) and len(ib) and ia[0] < ib[-1]:
                pa_, pb_ = ia[0], ib[-1]
            else:
                continue
            rows["eventA"].append(activity_names[a])
            rows["eventB"].append(activity_names[b])
            rows["trace_id"].append(trace_ids[t])
            rows["positionA"].append(int(pa_))
            rows["positionB"].append(int(pb_))
    return pa.table({"eventA": pa.array(rows["eventA"], type=pa.string()), "eventB": pa.array(rows["eventB"], type=pa.string()),
                     "trace_id": pa.array(rows["trace_id"], type=pa.string()),
                     "positionA": pa.array(rows["positionA"], type=pa.int32()),
                     "positionB": pa.array(rows["positionB"], type=pa.int32())})
