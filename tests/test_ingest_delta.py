"""Appending a batch of seq.parquet rows to a log (ingest.read_seq_delta + ingest.merge_delta): the merged log equals
the log read from the base and the batch as one table - same trace and activity numbering, case folding, new names,
unordered positions - and a batch that rewrites an existing position is refused."""
import numpy as np
import pyarrow as pa
import pytest

from sequencedetectionqueryexecutor_b200 import ingest
from sequencedetectionqueryexecutor_b200.sase import ActivityDictionary
from tests import gen


def _base(n_traces=120, seed=3):
    """seq.parquet rows of a random log and the log read back (a trace without events has no row, so it is absent)."""
    off, act, ts = gen.make_log(n_traces, 0, 12, 6, seed=seed, jitter_ms=True)
    names = ["Register", "approve", "Reject", "PAY", "ship", "close"]
    tb = ingest.seq_table_from_csr(off, act, ts, [f"case-{i:04d}" for i in range(n_traces)], names)
    return tb, ingest.read_seq_table(tb)


def _batch_table(off, ts, tids, seed):
    """Rows for some existing traces (positions continuing after their events, rows shuffled, a few ties) and for new
    traces; event names mix known ones in other cases with new ones."""
    rng = np.random.default_rng(seed)
    T = len(off) - 1
    names = ["register", "APPROVE", "audit", "Audit", "escalate", "pay"]
    rows = []
    for t in sorted(rng.choice(T, size=T // 3, replace=False)):
        n0 = int(off[t + 1] - off[t])
        t_last = int(ts[off[t + 1] - 1]) if n0 else gen.T0_MS
        for j in range(int(rng.integers(1, 5))):
            pos = n0 + j if rng.random() < 0.8 else n0            # ties on the first new position: table order decides
            rows.append((tids[t], names[int(rng.integers(0, len(names)))], t_last + 1000 * (j + 1), pos))
    for n in range(7):
        tid = f"new-{n}"
        for j in range(int(rng.integers(0, 6))):
            rows.append((tid, names[int(rng.integers(0, len(names)))], gen.T0_MS + 5000 * j, j))
    rng.shuffle(rows)
    ts_col = ingest._format_ts(np.array([r[2] for r in rows], dtype=np.int64))
    return pa.table({"trace_id": pa.array([r[0] for r in rows], type=pa.string()),
                     "event_type": pa.array([r[1] for r in rows], type=pa.string()),
                     "timestamp": pa.array(ts_col, type=pa.string()),
                     "position": pa.array([r[3] for r in rows], type=pa.int32())})


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_merge_of_the_delta_equals_reading_base_and_batch_together(seed):
    base_tb, base = _base(seed=seed + 10)
    batch_tb = _batch_table(base.trace_off, base.ts_ms, base.trace_ids, seed)
    whole = ingest.read_seq_table(pa.concat_tables([base_tb, batch_tb]))
    T = base.n_traces
    trace_ids = list(base.trace_ids)
    delta = ingest.read_seq_delta(batch_tb, trace_ids, base.activities, trace_lens=np.diff(base.trace_off))
    m_off, m_act, m_ts = ingest.merge_delta(base.trace_off, base.act, base.ts_ms, delta)

    assert trace_ids == whole.trace_ids
    assert base.activities.names == whole.activities.names
    assert delta.n_activities == len(whole.activities) and delta.n_new_traces == len(trace_ids) - T
    assert np.all(np.diff(delta.trace_idx) > 0)
    assert np.array_equal(m_off, whole.trace_off)
    assert np.array_equal(m_act, whole.act)
    assert np.array_equal(m_ts, whole.ts_ms)


def test_merge_delta_equals_a_per_trace_restatement():
    rng = np.random.default_rng(7)
    off, act, ts = gen.make_log(300, 0, 9, 5, seed=4)
    T, n_new = len(off) - 1, 40
    listed = np.sort(rng.choice(T + n_new, size=150, replace=False))
    lens = rng.integers(0, 4, size=len(listed))
    b_off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    b_act = rng.integers(0, 9, size=int(b_off[-1])).astype(np.int32)
    b_ts = rng.integers(0, 1 << 40, size=int(b_off[-1])).astype(np.int64)
    delta = ingest.SeqDelta(listed.astype(np.int64), b_off, b_act, b_ts, n_new, 9)
    m_off, m_act, m_ts = ingest.merge_delta(off, act, ts, delta)
    want_act, want_ts = [[] for _ in range(T + n_new)], [[] for _ in range(T + n_new)]
    for t in range(T):
        want_act[t] += list(act[off[t]:off[t + 1]])
        want_ts[t] += list(ts[off[t]:off[t + 1]])
    for i, t in enumerate(listed):
        want_act[t] += list(b_act[b_off[i]:b_off[i + 1]])
        want_ts[t] += list(b_ts[b_off[i]:b_off[i + 1]])
    assert np.array_equal(np.diff(m_off), [len(x) for x in want_act])
    assert m_act.tolist() == [int(v) for x in want_act for v in x]
    assert m_ts.tolist() == [int(v) for x in want_ts for v in x]
    # an empty batch changes nothing
    empty = ingest.SeqDelta(np.zeros(0, np.int64), np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int64), 0, 5)
    e_off, e_act, e_ts = ingest.merge_delta(off, act, ts, empty)
    assert np.array_equal(e_off, off) and np.array_equal(e_act, act) and np.array_equal(e_ts, ts)


def test_a_batch_that_rewrites_a_position_is_refused():
    _, base = _base(n_traces=20, seed=5)
    tids = base.trace_ids
    t = int(np.argmax(np.diff(base.trace_off)))                     # a trace that holds events
    n0 = int(base.trace_off[t + 1] - base.trace_off[t])
    tb = pa.table({"trace_id": [tids[t], tids[t]], "event_type": ["ship", "ship"],
                   "timestamp": ["2020-03-01 00:00:00", "2020-03-01 00:00:01"], "position": pa.array([n0, n0 - 1], type=pa.int32())})
    with pytest.raises(ValueError, match="not an append"):
        ingest.read_seq_delta(tb, list(base.trace_ids), ActivityDictionary(base.activities.names), trace_lens=np.diff(base.trace_off))
    # without the lengths the batch is taken as it is (the caller vouches for the positions)
    d = ingest.read_seq_delta(tb, list(base.trace_ids), ActivityDictionary(base.activities.names))
    assert d.trace_idx.tolist() == [t] and d.batch_off.tolist() == [0, 2] and d.n_new_traces == 0


def test_an_empty_batch():
    d = ingest.read_seq_delta(pa.table({"trace_id": pa.array([], pa.string()), "event_type": pa.array([], pa.string()),
                                        "timestamp": pa.array([], pa.string()), "position": pa.array([], pa.int32())}),
                              ["a"], ActivityDictionary(["x", "y"]))
    assert len(d.trace_idx) == 0 and d.batch_off.tolist() == [0] and d.n_new_traces == 0 and d.n_activities == 2
