"""Growing a resident log on the device (csrc/append.cu): siesta_log_append's columns equal ingest.merge_delta, and every
request on the appended log answers exactly as on a log loaded from the merged arrays."""
import threading

import numpy as np
import pytest

from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200 import ingest
from tests import gen

pytestmark = pytest.mark.gpu
N_, P_, S_, X_, O_ = abi.STATE_NORMAL, abi.STATE_KLEENE_PLUS, abi.STATE_KLEENE_STAR, abi.STATE_NEGATIVE, abi.STATE_OR

# NK class on kernel K1-P (the configs[4] shape), FK2 (a+ b* within), NP1 (a b* c), and a shape with a negation and a
# constrained OR state that runs on the run-list engine
NFAS = {
    "nk_k1p": [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
               dict(kind=X_, types=[3]), dict(kind=N_, types=[4]), dict(kind=N_, types=[5], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])],
    "fk2": [dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])],
    "np1": [dict(kind=N_, types=[0]), dict(kind=S_, types=[1]), dict(kind=N_, types=[2])],
    "engine": [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 900)]),
               dict(kind=X_, types=[3]), dict(kind=P_, types=[4])],
}


def rand_batch(rng, off, ts, n_new, n_listed, max_len, n_act, listed=None, act_hi=None):
    """A random batch whose timestamps keep every trace sorted: listed traces (ascending) out of T + n_new."""
    T = len(off) - 1
    if listed is None:
        listed = np.sort(rng.choice(T + n_new, size=min(n_listed, T + n_new), replace=False))
    listed = np.asarray(listed, dtype=np.int64)
    lens = rng.integers(0, max_len + 1, size=len(listed))
    b_off = np.zeros(len(listed) + 1, dtype=np.int64)
    np.cumsum(lens, out=b_off[1:])
    b_act = rng.integers(0, act_hi or n_act, size=int(b_off[-1])).astype(np.int32)
    b_ts = np.zeros(int(b_off[-1]), dtype=np.int64)
    for i, t in enumerate(listed):
        last = int(ts[off[t + 1] - 1]) if t < T and off[t + 1] > off[t] else gen.T0_MS
        b_ts[b_off[i]:b_off[i + 1]] = last + np.cumsum(rng.integers(0, 300, size=int(lens[i]))) * 1000
    return ingest.SeqDelta(listed, b_off, b_act, b_ts, n_new, n_act)


def _append(log, d, n_activities=None):
    return log.append(d.trace_idx, d.batch_off, d.act, d.ts_ms, d.n_new_traces, n_activities or d.n_activities)


def _columns_equal(log, want):
    off, act, ts = log.read()
    assert np.array_equal(off, want[0]) and np.array_equal(act, want[1]) and np.array_equal(ts, want[2])


def _same_detect(a, b, flags):
    for name, states in NFAS.items():
        nfa = abi.make_nfa(states)
        ok, why = a.detect(nfa, flags=flags).same_as(b.detect(nfa, flags=flags))
        assert ok, (name, flags, why)


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


CASES = ["random", "first_last", "empty_traces_gain", "new_listed_unlisted", "empty_batch", "every_trace", "many_new"]


@pytest.mark.parametrize("case", CASES)
def test_appended_columns_equal_merge_delta(ctx, case):
    rng = np.random.default_rng(CASES.index(case))
    min_len = 0 if case == "empty_traces_gain" else 1
    off, act, ts = gen.make_log(3000, min_len, 50, 12, seed=40 + CASES.index(case))
    T = len(off) - 1
    if case == "random":
        d = rand_batch(rng, off, ts, 0, 700, 9, 12)
    elif case == "first_last":
        d = rand_batch(rng, off, ts, 0, 0, 7, 12, listed=[0, 1, T // 2, T - 1])
    elif case == "empty_traces_gain":
        empty = np.flatnonzero(np.diff(off) == 0)
        assert len(empty) > 10
        d = rand_batch(rng, off, ts, 0, 0, 6, 12, listed=np.union1d(empty, [0, 5, 17]))
    elif case == "new_listed_unlisted":
        d = rand_batch(rng, off, ts, 50, 0, 6, 12, listed=np.concatenate((np.arange(3, T, 97), T + np.arange(0, 50, 3))))
    elif case == "empty_batch":
        d = rand_batch(rng, off, ts, 0, 0, 0, 12, listed=[])
    elif case == "every_trace":
        d = rand_batch(rng, off, ts, 0, T, 4, 12)
    else:   # thousands of new traces back to back: batch runs that cross tile boundaries
        d = rand_batch(rng, off, ts, 4000, 0, 12, 12, listed=np.concatenate(([2, 9], T + np.arange(4000))))
    want = ingest.merge_delta(off, act, ts, d)
    log = ctx.load_log(off, act, ts, 12)
    new, ms = _append(log, d)
    assert ms >= 0 and (new.n_traces, new.n_events) == (len(want[0]) - 1, len(want[1]))
    _columns_equal(new, want)
    # partial reads: offsets as stored, events of the range
    for t0, t1 in ((0, 1), (5, 900), (T - 3, new.n_traces), (new.n_traces, new.n_traces)):
        o, a, s = new.read(t0, t1)
        assert np.array_equal(o, want[0][t0:t1 + 1])
        assert np.array_equal(a, want[1][want[0][t0]:want[0][t1]]) and np.array_equal(s, want[2][want[0][t0]:want[0][t1]])
    new.close()
    log.close()


def test_requests_on_the_appended_log_equal_a_fresh_load(ctx):
    rng = np.random.default_rng(11)
    off, act, ts = gen.make_log(4000, 20, 60, 8, seed=12, max_gap_s=120)
    d = rand_batch(rng, off, ts, 300, 1500, 8, 8)
    want = ingest.merge_delta(off, act, ts, d)
    log = ctx.load_log(off, act, ts, 8)
    new, _ = _append(log, d)
    ref = ctx.load_log(*want, 8)
    for flags in (0, abi.F_RETURN_ALL):
        _same_detect(new, ref, flags)
    assert np.array_equal(new.declare_counts(40).packed, ref.declare_counts(40).packed)
    pairs = [(0, 1), (2, 3), (5, 5), (7, 0)]
    assert new.pair_stats(pairs)[0] == ref.pair_stats(pairs)[0]
    c1, d1, _ = new.explore_accurate([0, 1], list(range(8)))
    c2, d2, _ = ref.explore_accurate([0, 1], list(range(8)))
    assert np.array_equal(c1, c2) and np.array_equal(d1, d2)
    wnm = ([0, 1, 2], [(0, 1, abi.WNM_TIME, abi.WNM_WITHIN, 300), (1, 2, abi.WNM_TIME, abi.WNM_ATLEAST, 200)], 120, 60, 120)
    cand = np.arange(0, new.n_traces, 37, dtype=np.int64)
    ok, why = new.why_not_match(*wnm, cand=cand).same_as(ref.why_not_match(*wnm, cand=cand))
    assert ok, why
    lo, hi = int(want[2].min()), int(want[2].max())
    v1, v2 = new.filter_time(lo + (hi - lo) // 3, hi - (hi - lo) // 4), ref.filter_time(lo + (hi - lo) // 3, hi - (hi - lo) // 4)
    assert all(np.array_equal(x, y) for x, y in zip(v1.read(), v2.read()))
    _same_detect(v1, v2, 0)
    i1, i2 = new.build_index(pairs), ref.build_index(pairs)
    assert np.array_equal(i1.intersect([0, 1]), i2.intersect([0, 1]))
    for x in (i1, i2, v1, v2, new, ref, log):
        x.close()


def test_declare_counts_after_the_longest_trace_passes_64_and_128(ctx):
    rng = np.random.default_rng(3)
    off, act, ts = gen.make_log(2000, 30, 60, 20, seed=5)
    log = ctx.load_log(off, act, ts, 20)
    cur = (off, act, ts)
    for target in (70, 140):
        t = int(rng.integers(0, 2000))
        n0 = int(cur[0][t + 1] - cur[0][t])
        d = rand_batch(rng, *cur[::2], 0, 0, 1, 20, listed=[t])
        d.batch_off[1] = target - n0
        d.act = rng.integers(0, 20, size=target - n0).astype(np.int32)
        d.ts_ms = int(cur[2][cur[0][t + 1] - 1]) + np.arange(1, target - n0 + 1, dtype=np.int64) * 1000
        new, _ = _append(log, d)
        cur = ingest.merge_delta(*cur, d)
        ref = ctx.load_log(*cur, 20)
        assert np.array_equal(new.declare_counts(64).packed, ref.declare_counts(64).packed), target
        _same_detect(new, ref, 0)
        ref.close()
        log.close()
        log = new
    log.close()


@pytest.mark.parametrize("n_act_new", [33, 105, 256])
def test_growing_alphabet_takes_the_path_of_a_fresh_load(ctx, n_act_new):
    rng = np.random.default_rng(n_act_new)
    off, act, ts = gen.make_log(2500, 5, 40, 20, seed=9)
    d = rand_batch(rng, off, ts, 100, 900, 10, n_act_new)
    d.act[::7] = n_act_new - 1                                 # the new top id certainly occurs
    want = ingest.merge_delta(off, act, ts, d)
    log = ctx.load_log(off, act, ts, 20)
    new, _ = _append(log, d)
    ref = ctx.load_log(*want, n_act_new)
    _columns_equal(new, want)
    states = [dict(kind=N_, types=[0]), dict(kind=O_, types=[n_act_new - 1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
              dict(kind=X_, types=[3]), dict(kind=N_, types=[n_act_new - 2])]
    for flags in (0, abi.F_RETURN_ALL):
        _same_detect(new, ref, flags)
        ok, why = new.detect(abi.make_nfa(states), flags=flags).same_as(ref.detect(abi.make_nfa(states), flags=flags))
        assert ok, why
    assert np.array_equal(new.declare_counts(16).packed, ref.declare_counts(16).packed)
    for x in (new, ref, log):
        x.close()


def test_an_out_of_range_id_answers_as_a_load_of_that_id(ctx):
    rng = np.random.default_rng(4)
    off, act, ts = gen.make_log(1500, 5, 40, 10, seed=19)
    d = rand_batch(rng, off, ts, 20, 400, 6, 10)
    d.act[::5] = 13                                            # outside [0, 10)
    want = ingest.merge_delta(off, act, ts, d)
    log = ctx.load_log(off, act, ts, 10)
    new, _ = _append(log, d)
    ref = ctx.load_log(*want, 10)
    for flags in (0, abi.F_RETURN_ALL):
        _same_detect(new, ref, flags)
    assert np.array_equal(new.declare_counts(20).packed, ref.declare_counts(20).packed)
    for x in (new, ref, log):
        x.close()


def test_five_chained_appends_equal_one_load_and_old_handles_stay_valid(ctx):
    rng = np.random.default_rng(8)
    off, act, ts = gen.make_log(2000, 1, 40, 8, seed=31)
    nfa = abi.make_nfa(NFAS["nk_k1p"])
    log = ctx.load_log(off, act, ts, 8)
    before = log.detect(nfa, flags=abi.F_RETURN_ALL)
    cur, handles = (off, act, ts), [log]
    for i in range(5):
        d = rand_batch(rng, *cur[::2], 30 * i, 300, 8, 8)
        new, _ = _append(handles[-1], d)
        cur = ingest.merge_delta(*cur, d)
        handles.append(new)
    ok, why = log.detect(nfa, flags=abi.F_RETURN_ALL).same_as(before)      # the first handle answers as before
    assert ok, why
    _columns_equal(log, (off, act, ts))
    for h in handles[:-1]:
        h.close()                                                          # freeing the old ones leaves the last intact
    ref = ctx.load_log(*cur, 8)
    _columns_equal(handles[-1], cur)
    for flags in (0, abi.F_RETURN_ALL):
        _same_detect(handles[-1], ref, flags)
    ref.close()
    handles[-1].close()


def test_wrapped_base_and_shard_indices(ctx):
    import torch
    rng = np.random.default_rng(21)
    off, act, ts = gen.make_log(1800, 1, 30, 6, seed=2)
    d = rand_batch(rng, off, ts, 40, 500, 5, 6)
    want = ingest.merge_delta(off, act, ts, d)
    dev = torch.device("cuda", 0)
    tens = [torch.from_numpy(x).to(dev) for x in (off, act, ts)]
    wrapped = ctx.wrap_log(*tens, 6, max_trace_len=30)
    new, _ = _append(wrapped, d)
    wrapped.close()
    del tens
    _columns_equal(new, want)
    ref = ctx.load_log(*want, 6)
    _same_detect(new, ref, 0)
    new.close()
    # a shard keeps reporting global trace indices
    shard = ctx.load_log(off, act, ts, 6)
    shard.set_first_trace(1_000_000)
    ref.set_first_trace(1_000_000)
    new, _ = _append(shard, d)
    for flags in (0, abi.F_RETURN_ALL):
        _same_detect(new, ref, flags)
    assert new.detect(abi.make_nfa(NFAS["np1"])).trace_idx.min() >= 1_000_000
    for x in (new, shard, ref):
        x.close()


def test_detect_on_the_old_handle_while_appending(ctx):
    rng = np.random.default_rng(6)
    off, act, ts = gen.make_log(20000, 10, 60, 8, seed=7)
    log = ctx.load_log(off, act, ts, 8)
    nfa = abi.make_nfa(NFAS["engine"])
    want = log.detect(nfa, flags=abi.F_RETURN_ALL)
    errors, stop = [], threading.Event()

    def reader():
        n = 0
        while not stop.is_set() or n < 3:
            ok, why = log.detect(nfa, flags=abi.F_RETURN_ALL).same_as(want)
            if not ok:
                errors.append(why)
            n += 1

    th = threading.Thread(target=reader)
    th.start()
    try:
        for i in range(6):
            d = rand_batch(rng, off, ts, 100, 3000, 8, 8)
            new, _ = _append(log, d)
            _columns_equal(new, ingest.merge_delta(off, act, ts, d))
            new.close()
    finally:
        stop.set()
        th.join()
    assert not errors, errors
    log.close()


def test_invalid_batches_fail_and_leave_the_log_usable(ctx):
    from sequencedetectionqueryexecutor_b200 import api
    from sequencedetectionqueryexecutor_b200._lib import SiestaError
    off, act, ts = gen.make_log(200, 1, 20, 6, seed=1)
    log = ctx.load_log(off, act, ts, 6)
    nfa = abi.make_nfa(NFAS["np1"])
    want = log.detect(nfa)
    one_a, one_t = np.array([1], np.int32), np.array([gen.T0_MS + 10**9], np.int64)
    bad = {
        "descending": ([5, 3], [0, 1, 1], [1], [gen.T0_MS + 10**9]),
        "repeated": ([4, 4], [0, 0, 1], one_a, one_t),
        "negative": ([-1], [0, 1], one_a, one_t),
        "past_the_end": ([200], [0, 1], one_a, one_t),
        "off_not_from_0": ([3], [1, 1], one_a, one_t),
        "off_decreasing": ([3, 4], [0, 2, 1], one_a, one_t),
    }
    for name, (ti, bo, a, t) in bad.items():
        with pytest.raises(SiestaError) as ei:
            log.append(ti, bo, a, t)
        assert ei.value.code == abi.E_INVALID and "siesta_log_append" in str(ei.value), name
    # batch_off must end at the arrays' length: the library copies batch_off[-1] events from them
    for over_or_short in ([0, 5], [0, 0]):
        with pytest.raises(ValueError, match="batch_off"):
            log.append([3], over_or_short, one_a, one_t)
    with pytest.raises(SiestaError) as ei:
        log.append([3], [0, 1], one_a, one_t, n_new_traces=-1)
    assert ei.value.code == abi.E_INVALID
    with pytest.raises(SiestaError) as ei:
        log.append([3], [0, 1], one_a, one_t, n_activities=5)            # the dictionary only grows
    assert ei.value.code == abi.E_INVALID
    view = log.filter_time(None, None)
    with pytest.raises(SiestaError) as ei:
        view.append([3], [0, 1], one_a, one_t)                          # derived logs are per-request views
    assert ei.value.code == abi.E_INVALID
    view.close()
    blk = ctx.load_log(off, act, ts, 6)
    blk.set_blocks([0, 100, 200], [0, 1000])
    with pytest.raises(SiestaError) as ei:
        blk.append([3], [0, 1], one_a, one_t)                           # block-cyclic shard
    assert ei.value.code == abi.E_INVALID
    blk.close()
    import ctypes as C
    from sequencedetectionqueryexecutor_b200._lib import lib
    h = C.c_void_p()
    bo = np.array([0, 1], np.int64)
    rc = lib().siesta_log_append(log._h, None, api._ptr(bo), 1, api._ptr(one_a), api._ptr(one_t), 0, 6, C.byref(h), None)
    assert rc == abi.E_INVALID and not h.value and lib().siesta_last_error()
    rc = lib().siesta_log_append(log._h, api._ptr(np.array([3], np.int64)), api._ptr(bo), 1, None, None, 0, 6, C.byref(h), None)
    assert rc == abi.E_INVALID and not h.value
    ok, why = log.detect(nfa).same_as(want)
    assert ok, why
    _columns_equal(log, (off, act, ts))
    log.close()


def test_multi_log_append_equals_a_multi_load_of_the_merged_log():
    from sequencedetectionqueryexecutor_b200 import api
    rng = np.random.default_rng(17)
    off, act, ts = gen.make_log(3000, 1, 50, 8, seed=23, max_gap_s=120)
    d = rand_batch(rng, off, ts, 200, 1200, 8, 10)
    d.act[::11] = 9                                                     # the alphabet grows as well
    want = ingest.merge_delta(off, act, ts, d)
    with api.Multi([0, 0]) as m:
        ml = m.load_log(off, act, ts, 8)
        before = ml.detect(abi.make_nfa(NFAS["fk2"]))
        new = ml.append(d.trace_idx, d.batch_off, d.act, d.ts_ms, d.n_new_traces, 10)
        ref = m.load_log(*want, 10)
        for flags in (0, abi.F_RETURN_ALL):
            for name, states in NFAS.items():
                ok, why = new.detect(abi.make_nfa(states), flags=flags).same_as(ref.detect(abi.make_nfa(states), flags=flags))
                assert ok, (name, flags, why)
        assert np.array_equal(new.declare_counts(30).packed, ref.declare_counts(30).packed)
        wnm = ([0, 1, 2], [(0, 1, abi.WNM_TIME, abi.WNM_WITHIN, 300)], 120, 60, 120)
        cand = np.arange(0, 3200, 29, dtype=np.int64)
        ok, why = new.why_not_match(*wnm, cand=cand).same_as(ref.why_not_match(*wnm, cand=cand))
        assert ok, why
        with pytest.raises(ValueError, match="batch_off"):
            ml.append(d.trace_idx, d.batch_off + np.arange(len(d.batch_off)), d.act, d.ts_ms, d.n_new_traces, 10)
        ok, why = ml.detect(abi.make_nfa(NFAS["fk2"])).same_as(before)   # the old multi log is unchanged
        assert ok, why
        for x in (new, ref, ml):
            x.close()
