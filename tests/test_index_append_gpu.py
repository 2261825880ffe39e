"""A pair index that follows a growing log (csrc/intersect.cu): PairIndex.refresh equals a rebuild on the appended log and
the oracle's SeqTable-view lists, PairIndex.append equals a load of the union lists, and intersect / candidates on the
results equal those on the reference indexes, bit for bit."""
import ctypes as C
import threading

import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200 import ingest
from sequencedetectionqueryexecutor_b200.sase import ActivityDictionary
from tests import gen
from tests.test_log_append_gpu import rand_batch

pytestmark = pytest.mark.gpu

N_ACT = 10
PAIRS = [(0, 1), (2, 3), (5, 5), (7, 0), (1, 4), (3, 3), (9, 8)]
EXPANSIONS = [[0, 1], [2, 3, 4], [5], [0, 2, 6]]
SCAN_CHUNK = 1024 * 256   # row_scan_kernel scans 1 024 block counts of 256 flags per pass


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


def _append(log, d):
    return log.append(d.trace_idx, d.batch_off, d.act, d.ts_ms, d.n_new_traces, d.n_activities)


def _lists(ix):
    return [ix.posting_list(i) for i in range(len(ix.pairs))]


def _oracle(off, act, pairs):
    return [oracle.posting_list(off, act, a, b) for a, b in pairs]


def _same_lists(got, want, what=""):
    assert len(got) == len(want), what
    for p, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == np.int64 and np.array_equal(g, w), (what, p, len(g), len(w))


def _answers(ix):
    n = len(ix.pairs)
    out = [ix.intersect(ids) for ids in ([0], [0, 1], [1, 2, 3], list(range(n)))]
    return out + [ix.candidates([x for x in EXPANSIONS if max(x) < n])]


def _same_answers(a, b):
    for i, (x, y) in enumerate(zip(_answers(a), _answers(b))):
        assert np.array_equal(x, y), i


def _batch_delta(new_off, new_act, listed, pairs, n_act):
    """The batch's index.parquet rows (written for its listed traces on the grown log) read back with
    ingest.read_index_table and aligned with `pairs`."""
    names = [f"Act{i}" for i in range(n_act)]
    tids = [f"trace-{t}" for t in range(len(new_off) - 1)]
    listed = np.asarray(listed, dtype=np.int64)
    lens = np.diff(new_off)[listed]
    sub_off = np.zeros(len(listed) + 1, dtype=np.int64)
    np.cumsum(lens, out=sub_off[1:])
    sub_act = (np.concatenate([new_act[new_off[t]:new_off[t + 1]] for t in listed]) if len(listed)
               else np.zeros(0, dtype=np.int32))
    tb = ingest.index_table_from_csr(sub_off, sub_act, [tids[t] for t in listed], names, pairs)
    seq = ingest.SeqLog(new_off, new_act, np.zeros(len(new_act), np.int64), tids, ActivityDictionary(names))
    got_pairs, lists = ingest.read_index_table(tb, seq, [(names[a], names[b]) for a, b in pairs])
    by_pair = dict(zip(got_pairs, lists))
    return [by_pair.get(p, np.zeros(0, dtype=np.int64)) for p in pairs]


def _with_new(rng, off, ts, n_new, n_touched, max_len, n_act):
    """rand_batch whose listed traces hold every new trace (a seq.parquet batch lists each trace it adds)."""
    T = len(off) - 1
    touched = np.sort(rng.choice(T, size=min(n_touched, T), replace=False))
    return rand_batch(rng, off, ts, n_new, 0, max_len, n_act, listed=np.concatenate((touched, T + np.arange(n_new))))


BATCHES = ["touched", "new", "both", "empty", "every"]


@pytest.mark.parametrize("case", BATCHES)
def test_refresh_and_append_follow_a_random_batch(ctx, case):
    rng = np.random.default_rng(100 + BATCHES.index(case))
    off, act, ts = gen.make_log(3000, 0, 24, N_ACT, seed=60 + BATCHES.index(case))
    T = len(off) - 1
    if case == "touched":
        d = _with_new(rng, off, ts, 0, 700, 6, N_ACT)
    elif case == "new":
        d = _with_new(rng, off, ts, 250, 0, 12, N_ACT)
    elif case == "both":
        d = _with_new(rng, off, ts, 150, 900, 8, N_ACT)
    elif case == "empty":
        d = rand_batch(rng, off, ts, 0, 0, 0, N_ACT, listed=[])
    else:
        d = _with_new(rng, off, ts, 0, T, 4, N_ACT)
    w_off, w_act, w_ts = ingest.merge_delta(off, act, ts, d)
    want = _oracle(w_off, w_act, PAIRS)
    log = ctx.load_log(off, act, ts, N_ACT)
    new, _ = _append(log, d)
    # built index -> refresh == siesta_index_build on the new log == the oracle
    built = log.build_index(PAIRS)
    old_lists, old_answers = _lists(built), _answers(built)
    ref, ms = built.refresh(new, d.trace_idx)
    assert ms >= 0 and ref.log is new and ref.pairs == built.pairs
    rebuilt = new.build_index(PAIRS)
    _same_lists(_lists(rebuilt), want, "build")
    _same_lists(_lists(ref), want, "refresh")
    _same_answers(ref, rebuilt)
    # loaded index -> append of the batch's index.parquet rows == load of the union lists
    loaded = log.load_index(PAIRS, _oracle(off, act, PAIRS))
    delta = _batch_delta(w_off, w_act, d.trace_idx, PAIRS, N_ACT)
    union = [np.union1d(o, x).astype(np.int64) for o, x in zip(_oracle(off, act, PAIRS), delta)]
    _same_lists(union, want, "union of the old lists and the batch's rows")
    app, ms = loaded.append(new, delta)
    assert ms >= 0
    reloaded = new.load_index(PAIRS, union)
    _same_lists(_lists(app), union, "append")
    _same_answers(app, reloaded)
    _same_answers(app, rebuilt)
    # the old indexes answer as before
    _same_lists(_lists(built), old_lists, "old built index")
    for x, y in zip(_answers(built), old_answers):
        assert np.array_equal(x, y)
    _same_lists(_lists(loaded), old_lists, "old loaded index")
    for x in (built, ref, rebuilt, loaded, app, reloaded, new, log):
        x.close()


def test_append_merges_hand_made_edge_lists(ctx):
    """Inserts before the first and after the last old entry, a delta equal to its old list, an empty old list, empty
    deltas, long runs of inserts across pair boundaries and more than 32 pairs (a loaded index has no pair limit)."""
    off, act, ts = gen.make_log(600, 1, 10, N_ACT, seed=3)
    rng = np.random.default_rng(5)
    d = _with_new(rng, off, ts, 400, 0, 3, N_ACT)
    log = ctx.load_log(off, act, ts, N_ACT)
    new, _ = _append(log, d)
    T, T2 = log.n_traces, new.n_traces
    old = [np.array([5, 7, 9, 300]), np.array([], np.int64), np.array([2, 4, 599]), np.arange(0, T, 3),
           np.arange(T), np.array([10]), np.array([], np.int64)]
    dl = [np.array([0, 4, 6, 9, 12, 301, T2 - 1]), np.array([1, 2, 3, T + 5]), np.array([2, 4, 599]), np.array([], np.int64),
          np.arange(T, T2), np.arange(0, T2, 2), np.array([], np.int64)]
    rnd_old = [np.sort(rng.choice(T, size=int(rng.integers(0, T)), replace=False)) for _ in range(33)]
    rnd_dl = [np.sort(rng.choice(T2, size=int(rng.integers(0, 200)), replace=False)) for _ in range(33)]
    old, dl = old + rnd_old, dl + rnd_dl
    pairs = [(p % N_ACT, (p * 7) % N_ACT) for p in range(len(old))]
    ix = log.load_index(pairs, old)
    app, _ = ix.append(new, dl)
    want = [np.union1d(o, x).astype(np.int64) for o, x in zip(old, dl)]
    _same_lists(_lists(app), want)
    ref = new.load_index(pairs, want)
    for ids in ([0], [0, 2], [3, 4], [4, 5], list(range(32))):
        assert np.array_equal(app.intersect(ids), ref.intersect(ids))
    _same_lists(_lists(ix), [o.astype(np.int64) for o in old], "old index")
    # every delta empty: the lists move unchanged
    same, _ = ix.append(new, [np.zeros(0, np.int64)] * len(old))
    _same_lists(_lists(same), [o.astype(np.int64) for o in old])
    for x in (ix, app, ref, same, new, log):
        x.close()


def test_refresh_edge_cases(ctx):
    """(a, a) completed by the batch; an activity the batch adds to the alphabet; an empty trace and new traces that
    gain pairs; inserts into empty old lists, before the first and after the last old entry; pairs the batch does not
    change."""
    # traces [0 1] [1 2] [3 3] [] [2 1]; the batch: trace 0 += [0], trace 3 += [2 1], new traces [4 1] and [0 0 1]
    off = np.array([0, 2, 4, 6, 6, 8], np.int64)
    act = np.array([0, 1, 1, 2, 3, 3, 2, 1], np.int32)
    ts = gen.T0_MS + np.arange(8, dtype=np.int64) * 1000
    log = ctx.load_log(off, act, ts, 4)
    pairs = [(0, 0), (2, 1), (3, 3), (4, 1), (1, 4), (0, 1), (3, 2)]
    d = ingest.SeqDelta(np.array([0, 3, 5, 6], np.int64), np.array([0, 1, 3, 5, 8], np.int64),
                        np.array([0, 2, 1, 4, 1, 0, 0, 1], np.int32), gen.T0_MS + 10**6 + np.arange(8, dtype=np.int64), 2, 5)
    w_off, w_act, _ = ingest.merge_delta(off, act, ts, d)
    new, _ = _append(log, d)
    built = log.build_index(pairs)
    assert len(built.posting_list(0)) == 0 and len(built.posting_list(3)) == 0 and list(built.posting_list(1)) == [4]
    ref, _ = built.refresh(new, d.trace_idx)
    want = _oracle(w_off, w_act, pairs)
    assert list(want[0]) == [0, 6] and list(want[1]) == [3, 4] and list(want[3]) == [5] and list(want[5]) == [0, 6]
    _same_lists(_lists(ref), want)
    rebuilt = new.build_index(pairs)
    _same_lists(_lists(rebuilt), want)
    _same_answers(ref, rebuilt)
    for x in (built, ref, rebuilt, new, log):
        x.close()


@pytest.mark.parametrize("grow", [True, False])
def test_refresh_after_out_of_range_ids_equals_a_rebuild(ctx, grow):
    """The old log holds id 11 outside its alphabet of 10.  When the batch grows the alphabet over it, traces the batch
    did not list gain (11, x) pairs: refresh flags every trace again and still equals siesta_index_build."""
    rng = np.random.default_rng(7)
    off, act, ts = gen.make_log(2000, 2, 20, N_ACT, seed=8)
    act = act.copy()
    act[::9] = 11
    d = _with_new(rng, off, ts, 30, 200, 5, 12 if grow else N_ACT)
    log = ctx.load_log(off, act, ts, N_ACT)
    new, _ = _append(log, d)
    pairs = [(11, 1), (2, 11), (11, 11), (0, 1)]
    built = log.build_index(pairs)
    assert all(len(built.posting_list(p)) == 0 for p in range(3))   # id 11 is unknown to the old log
    ref, _ = built.refresh(new, d.trace_idx)
    rebuilt = new.build_index(pairs)
    _same_lists(_lists(ref), _lists(rebuilt))
    _same_answers(ref, rebuilt)
    got = ref.posting_list(0)
    if grow:
        w_off, w_act, _ = ingest.merge_delta(off, act, ts, d)
        _same_lists(_lists(ref), _oracle(w_off, w_act, pairs))
        assert len(np.setdiff1d(got, d.trace_idx)) > 100   # unlisted traces gained the pair
    else:
        assert len(got) == 0
    for x in (built, ref, rebuilt, new, log):
        x.close()


def test_scale_lists_and_deltas_past_one_scan_chunk(ctx):
    """About 300 000 traces, a batch that lists more than 262 144 of them: the refresh's compaction carries in
    row_scan_kernel, the merge's delta scan runs past one chunk and its grid spans many blocks."""
    rng = np.random.default_rng(77)
    off, act, ts = gen.make_log(300_007, 1, 12, N_ACT, seed=78)
    d = _with_new(rng, off, ts, 3001, 280_000, 4, N_ACT)
    assert len(d.trace_idx) > SCAN_CHUNK
    w_off, w_act, _ = ingest.merge_delta(off, act, ts, d)
    want = _oracle(w_off, w_act, PAIRS)
    log = ctx.load_log(off, act, ts, N_ACT)
    new, _ = _append(log, d)
    built = log.build_index(PAIRS)
    ref, _ = built.refresh(new, d.trace_idx)
    _same_lists(_lists(ref), want)
    rebuilt = new.build_index(PAIRS)
    _same_answers(ref, rebuilt)
    old = _oracle(off, act, PAIRS)
    delta = [np.intersect1d(w, d.trace_idx).astype(np.int64) for w in want]
    assert sum(len(x) for x in delta) > SCAN_CHUNK
    loaded = log.load_index(PAIRS, old)
    app, _ = loaded.append(new, delta)
    _same_lists(_lists(app), want)
    _same_answers(app, rebuilt)
    for x in (built, ref, rebuilt, loaded, app, new, log):
        x.close()


def test_three_chained_refreshes_equal_one_build(ctx):
    rng = np.random.default_rng(12)
    off, act, ts = gen.make_log(2500, 1, 20, N_ACT, seed=13)
    cur = (off, act, ts)
    log = ctx.load_log(off, act, ts, N_ACT)
    ix = log.build_index(PAIRS)
    logs, idxs = [log], [ix]
    for i in range(3):
        d = _with_new(rng, cur[0], cur[2], 40 * (i + 1), 500, 6, N_ACT)
        new, _ = _append(logs[-1], d)
        nx, _ = idxs[-1].refresh(new, d.trace_idx)
        cur = ingest.merge_delta(*cur, d)
        logs.append(new)
        idxs.append(nx)
    final = ctx.load_log(*cur, N_ACT)
    rebuilt = final.build_index(PAIRS)
    _same_lists(_lists(idxs[-1]), _lists(rebuilt))
    _same_lists(_lists(rebuilt), _oracle(cur[0], cur[1], PAIRS))
    _same_answers(idxs[-1], rebuilt)
    _same_lists(_lists(idxs[0]), _oracle(off, act, PAIRS), "first index")
    for x in idxs + [rebuilt, final] + logs:
        x.close()


def test_old_index_answers_while_another_thread_refreshes(ctx):
    rng = np.random.default_rng(21)
    off, act, ts = gen.make_log(20000, 5, 40, N_ACT, seed=22)
    log = ctx.load_log(off, act, ts, N_ACT)
    ix = log.build_index(PAIRS)
    want = _answers(ix)
    errors, stop = [], threading.Event()

    def reader():
        n = 0
        while not stop.is_set() or n < 3:
            got = _answers(ix)
            if not all(np.array_equal(x, y) for x, y in zip(got, want)):
                errors.append(n)
            n += 1

    th = threading.Thread(target=reader)
    th.start()
    try:
        for i in range(4):
            d = _with_new(rng, off, ts, 100, 3000, 6, N_ACT)
            new, _ = _append(log, d)
            nx, _ = ix.refresh(new, d.trace_idx)
            w_off, w_act, _ = ingest.merge_delta(off, act, ts, d)
            _same_lists(_lists(nx), _oracle(w_off, w_act, PAIRS))
            nx.close()
            new.close()
    finally:
        stop.set()
        th.join()
    assert not errors, errors
    for x, y in zip(_answers(ix), want):
        assert np.array_equal(x, y)
    ix.close()
    log.close()


def test_refused_calls_leave_the_index_as_it_was(ctx):
    from sequencedetectionqueryexecutor_b200 import api
    from sequencedetectionqueryexecutor_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(31)
    off, act, ts = gen.make_log(300, 1, 15, N_ACT, seed=32)
    log = ctx.load_log(off, act, ts, N_ACT)
    d = _with_new(rng, off, ts, 5, 40, 4, N_ACT)
    new, _ = _append(log, d)
    T, T2 = log.n_traces, new.n_traces
    built = log.build_index(PAIRS)
    loaded = log.load_index(PAIRS, _lists(built))
    want_lists, want_answers = _lists(built), _answers(built)
    n = len(PAIRS)
    i64 = lambda x: np.ascontiguousarray(x, dtype=np.int64)   # noqa: E731
    good_off = i64(np.arange(n + 1))
    good_flat = i64(np.full(n, T2 - 1))

    def app(ix, lg, doff, flat):
        h = C.c_void_p()
        rc = L.siesta_index_append(ix, lg, None if doff is None else api._ptr(doff), None if flat is None else api._ptr(flat),
                                   C.byref(h), None)
        return rc, h.value

    rc, h = app(loaded._h, new._h, good_off, good_flat)                 # the well-formed call is accepted
    assert rc == 0 and h
    L.siesta_index_free(h)
    other = api.Context(0)
    other_log = other.load_log(off, act, ts, N_ACT)
    small = ctx.load_log(off[:101], act[:off[100]], ts[:off[100]], N_ACT)
    bad_append = {
        "null index": (None, new._h, good_off, good_flat),
        "null log": (loaded._h, None, good_off, good_flat),
        "null offsets": (loaded._h, new._h, None, good_flat),
        "null entries": (loaded._h, new._h, good_off, None),
        "other context": (loaded._h, other_log._h, good_off, good_flat),
        "fewer traces": (loaded._h, small._h, good_off, i64(np.zeros(n))),
        "off not from 0": (loaded._h, new._h, i64([1] + list(range(1, n + 1))), good_flat),
        "off decreasing": (loaded._h, new._h, i64([0, 2, 1] + list(range(3, n + 1))), good_flat),
        "not ascending": (loaded._h, new._h, i64([0, 2] + [2] * (n - 1)), i64([7, 3])),
        "repeated": (loaded._h, new._h, i64([0, 2] + [2] * (n - 1)), i64([4, 4])),
        "negative": (loaded._h, new._h, good_off, i64([-1] + [0] * (n - 1))),
        "past the end": (loaded._h, new._h, good_off, i64([T2] + [0] * (n - 1))),
    }
    for name, (ix, lg, doff, flat) in bad_append.items():
        rc, h = app(ix, lg, doff, flat)
        assert rc == abi.E_INVALID and not h, name
        assert L.siesta_last_error(), name
    assert L.siesta_index_append(loaded._h, new._h, api._ptr(good_off), api._ptr(good_flat), None, None) == abi.E_INVALID
    ti = i64(d.trace_idx)
    new_only = i64(np.arange(T, T2))
    bad_refresh = {
        "loaded index": (loaded._h, new._h, ti, None),
        "appended index": (None, new._h, ti, None),   # filled in below: the result of an append counts as loaded
        "null log": (built._h, None, ti, None),
        "other context": (built._h, other_log._h, i64([]), 0),
        "fewer traces": (built._h, small._h, i64([]), 0),
        "negative count": (built._h, new._h, ti, -1),
        "null list": (built._h, new._h, None, 3),
        "not ascending": (built._h, new._h, i64(np.concatenate(([9, 3], new_only))), None),
        "repeated": (built._h, new._h, i64(np.concatenate(([3, 3], new_only))), None),
        "negative": (built._h, new._h, i64(np.concatenate(([-1], new_only))), None),
        "past the end": (built._h, new._h, i64(np.concatenate((new_only, [T2]))), None),
        "a new trace missing": (built._h, new._h, i64(np.concatenate(([3], new_only[1:]))), None),
        "no new trace": (built._h, new._h, i64([3, 4]), None),
    }
    appended, _ = built.append(new, [np.zeros(0, np.int64)] * n)
    bad_refresh["appended index"] = (appended._h, new._h, ti, None)
    for name, (ix, lg, t, k) in bad_refresh.items():
        h = C.c_void_p()
        rc = L.siesta_index_refresh(ix, lg, None if t is None else api._ptr(t), len(t) if k is None else k, C.byref(h), None)
        assert rc == abi.E_INVALID and not h.value, name
    with pytest.raises(ValueError, match="delta lists"):
        loaded.append(new, [np.zeros(0, np.int64)] * (n - 1))
    for ix in (built, loaded):
        _same_lists(_lists(ix), want_lists)
        for x, y in zip(_answers(ix), want_answers):
            assert np.array_equal(x, y)
    ok, _ = built.refresh(new, d.trace_idx)                     # and the index still refreshes
    w_off, w_act, _ = ingest.merge_delta(off, act, ts, d)
    _same_lists(_lists(ok), _oracle(w_off, w_act, PAIRS))
    for x in (ok, appended, built, loaded, small, other_log, new, log):
        x.close()
    other.close()
