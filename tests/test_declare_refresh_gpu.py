"""The /declare counts follow a growing log (csrc/declare.cu): EventLog.declare_counts_refresh after siesta_log_append equals
siesta_declare_counts on the appended log, bit for bit on the whole packed array, for every K3 kernel family, alphabet
growth, histogram edge and batch shape.  Each test checks from the torch.profiler kernel names that the refresh ran the
family it is about (work-list instantiations, `true`) and declare_merge_kernel, or the full count where it falls back.
The test bodies run in one worker process (fixture `child`), so the profiler never starts in the pytest process."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200 import ingest
from tests import gen

pytestmark = pytest.mark.gpu

HS = 16   # histogram buckets K3 keeps in shared memory


def rand_batch(rng, off, ts, n_new, n_listed, max_len, n_act, listed=None, act_hi=None, min_len=0):
    """A random batch whose timestamps keep every trace sorted: listed traces (ascending) out of T + n_new
    (the batch generator of tests/test_log_append_gpu.py, with a minimum batch length per listed trace)."""
    T = len(off) - 1
    if listed is None:
        listed = np.sort(rng.choice(T + n_new, size=min(n_listed, T + n_new), replace=False))
    listed = np.asarray(listed, dtype=np.int64)
    lens = rng.integers(min_len, max_len + 1, size=len(listed))
    b_off = np.zeros(len(listed) + 1, dtype=np.int64)
    np.cumsum(lens, out=b_off[1:])
    b_act = rng.integers(0, act_hi or n_act, size=int(b_off[-1])).astype(np.int32)
    b_ts = np.zeros(int(b_off[-1]), dtype=np.int64)
    for i, t in enumerate(listed):
        last = int(ts[off[t + 1] - 1]) if t < T and off[t + 1] > off[t] else gen.T0_MS
        b_ts[b_off[i]:b_off[i + 1]] = last + np.cumsum(rng.integers(0, 300, size=int(lens[i]))) * 1000
    return ingest.SeqDelta(listed, b_off, b_act, b_ts, n_new, n_act)


def with_new(rng, off, ts, n_new, n_touched, max_len, n_act, **kw):
    """rand_batch listing n_touched old traces and every one of n_new new traces."""
    T = len(off) - 1
    touched = np.sort(rng.choice(T, size=min(n_touched, T), replace=False))
    return rand_batch(rng, off, ts, n_new, 0, max_len, n_act, listed=np.concatenate((touched, T + np.arange(n_new))), **kw)


def _append(log, d, n_activities=None):
    return log.append(d.trace_idx, d.batch_off, d.act, d.ts_ms, d.n_new_traces, n_activities or d.n_activities)[0]


def _kernel_names(fn):
    """(fn(), names of the CUDA kernels it launched) from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _uses(names, pattern):
    return any(re.search(pattern, n) for n in names)


# work-list (refresh) and full-log instantiations of each family
PAIRS_WL = r"declare_pairs_kernel<{}, \d, true>"
SERIAL_WL = r"declare_kernel<{}, true>"
ALT_WL = r"declare_alt_chain_kernel<{}, true>"
ANY_WL = r"declare_any_kernel<true>"
MERGE = r"declare_merge_kernel"
FULL = r"declare_(pairs_|alt_chain_|any_)?kernel<(\d, )*false>"


@pytest.fixture(scope="module")
def child():
    """Runs each test's body in one worker process for the module.  torch.profiler (CUPTI) then never starts in the pytest
    process: started there, it hid the K1-P / K1-L kernels from the traces of a later module in the same process
    (tests/test_uniform_placement_gpu.py).  The worker ends with the module."""
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(1) as pool:
        yield lambda fn, *args, env=None: pool.apply(_run, (fn, args, env))


_CTX = []


def _run(fn, args, env):
    """In the worker: fn(ctx, *args) with the environment variable `env` set to 1 (None: none)."""
    if not _CTX:
        from sequencedetectionqueryexecutor_b200 import api
        _CTX.append(api.Context(0))
    old = os.environ.get(env) if env else None
    if env:
        os.environ[env] = "1"
    try:
        fn(_CTX[0], *args)
    finally:
        if env and old is None:
            del os.environ[env]
        elif env:
            os.environ[env] = old


def _refresh(ctx, off, act, ts, n_act, d, k_cap=40, n_act_new=None):
    """(refreshed counts, full count of the new log, kernel names of the refresh, old counts): the two must be equal."""
    log = ctx.load_log(off, act, ts, n_act)
    old = log.declare_counts(k_cap)
    new = _append(log, d, n_act_new)
    got, names = _kernel_names(lambda: new.declare_counts_refresh(log, old, d.trace_idx))
    want = new.declare_counts(k_cap)
    # the old log is only read: it still answers as before
    assert np.array_equal(log.declare_counts(k_cap).packed, old.packed)
    new.close()
    log.close()
    return got, want, names, old


def _same(got, want):
    assert got.n_activities == want.n_activities and got.packed.shape == want.packed.shape
    bad = np.flatnonzero(got.packed != want.packed)
    assert len(bad) == 0, f"{len(bad)} values differ, first at {bad[:8]}"


# ------------------------------------------------------------------------------------------------ kernel families
# (case, n_act, old trace lengths, batch events per listed trace, forced family, kernels the refresh must run)
FAMILIES = [
    ("pairs_w2", 20, (0, 50), (0, 10), None, [PAIRS_WL.format(2)]),
    ("pairs_w3", 20, (66, 80), (0, 12), None, [PAIRS_WL.format(3)]),
    ("pairs_w4", 32, (100, 115), (0, 12), None, [PAIRS_WL.format(4)]),
    ("serial_nb1_long", 20, (100, 140), (0, 10), None, [SERIAL_WL.format(1), ALT_WL.format(1)]),
    ("serial_nb2", 33, (0, 60), (0, 10), None, [SERIAL_WL.format(2), ALT_WL.format(2)]),
    ("serial_nb3", 80, (0, 60), (0, 10), None, [SERIAL_WL.format(3), ALT_WL.format(3)]),
    ("serial_nb4", 104, (0, 60), (0, 10), None, [SERIAL_WL.format(4), ALT_WL.format(4)]),
    ("any_105", 105, (0, 60), (0, 10), None, [ANY_WL]),
    ("any_600", 600, (0, 60), (0, 10), None, [ANY_WL]),
    ("forced_serial", 12, (0, 50), (0, 10), "SIESTA_K3_SERIAL", [SERIAL_WL.format(1), ALT_WL.format(1)]),
    ("forced_any", 12, (0, 50), (0, 10), "SIESTA_K3_ANY", [ANY_WL]),
]


@pytest.mark.parametrize("case,n_act,lens,blen,env,kernels", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_refresh_equals_full_count_per_family(child, case, n_act, lens, blen, env, kernels):
    child(_refresh_equals_full_count_per_family, case, n_act, lens, blen, env, kernels, env=env)


def _refresh_equals_full_count_per_family(ctx, case, n_act, lens, blen, env, kernels):
    i = [f[0] for f in FAMILIES].index(case)
    rng = np.random.default_rng(500 + i)
    off, act, ts = gen.make_log(2500, lens[0], lens[1], n_act, seed=510 + i)
    d = with_new(rng, off, ts, 40, 600, blen[1], n_act, min_len=blen[0])
    got, want, names, _ = _refresh(ctx, off, act, ts, n_act, d)
    _same(got, want)
    for k in kernels + [MERGE]:
        assert _uses(names, k), (k, sorted(names))
    assert not _uses(names, FULL), sorted(names)


def test_pair_counts_then_a_serial_delta_when_a_trace_crosses_128(child):
    child(_pair_counts_then_a_serial_delta_when_a_trace_crosses_128)


def _pair_counts_then_a_serial_delta_when_a_trace_crosses_128(ctx):
    """The old log's longest trace is 120 events: its counts come from the pair kernel.  The batch takes listed traces past
    128, so the delta of the new versions runs on the serial kernels and the one of the old versions on the pair kernel."""
    rng = np.random.default_rng(7)
    off, act, ts = gen.make_log(2000, 90, 120, 16, seed=8)
    log = ctx.load_log(off, act, ts, 16)
    old, names_old = _kernel_names(lambda: log.declare_counts(40))
    assert _uses(names_old, r"declare_pairs_kernel<4, \d, false>")
    d = with_new(rng, off, ts, 10, 300, 20, 16, min_len=10)
    new = _append(log, d)
    got, names = _kernel_names(lambda: new.declare_counts_refresh(log, old, d.trace_idx))
    _same(got, new.declare_counts(40))
    assert _uses(names, PAIRS_WL.format(4)) and _uses(names, SERIAL_WL.format(1)) and _uses(names, MERGE), sorted(names)
    new.close()
    log.close()


# ------------------------------------------------------------------------------------------------ batch shapes
BATCHES = ["random", "empty", "listed_no_events", "every_trace", "empty_trace_gains"]


@pytest.mark.parametrize("case", BATCHES)
def test_refresh_follows_batch_shapes(child, case):
    child(_refresh_follows_batch_shapes, case)


def _refresh_follows_batch_shapes(ctx, case):
    i = BATCHES.index(case)
    rng = np.random.default_rng(600 + i)
    off, act, ts = gen.make_log(3000, 0, 40, 14, seed=610 + i)
    T = len(off) - 1
    if case == "random":
        d = with_new(rng, off, ts, 120, 900, 8, 14)
    elif case == "empty":
        d = rand_batch(rng, off, ts, 0, 0, 0, 14, listed=[])
    elif case == "listed_no_events":   # listed traces that receive nothing, new traces that stay empty
        d = rand_batch(rng, off, ts, 30, 0, 0, 14, listed=np.concatenate((np.arange(0, T, 37), T + np.arange(30))))
    elif case == "every_trace":
        d = with_new(rng, off, ts, 0, T, 4, 14)
    else:   # old traces that were empty receive events: their first / last activity appears
        empty = np.flatnonzero(np.diff(off) == 0)
        assert len(empty) > 20
        d = rand_batch(rng, off, ts, 0, 0, 6, 14, listed=np.union1d(empty, [1, 2, 3]), min_len=1)
    got, want, names, old = _refresh(ctx, off, act, ts, 14, d)
    _same(got, want)
    assert _uses(names, MERGE) and not _uses(names, FULL), sorted(names)
    if case == "empty":
        assert np.array_equal(got.packed, old.packed)
    if case == "empty_trace_gains":
        assert (got.first != old.first).any() and got.n_nonempty > old.n_nonempty


# ------------------------------------------------------------------------------------------------ alphabet growth
GROWTH = [("32_to_33", 32, 33, [PAIRS_WL.format(2)], [SERIAL_WL.format(2)]), ("104_to_105", 104, 105, [SERIAL_WL.format(4)], [ANY_WL])]


@pytest.mark.parametrize("case,a0,a1,old_kernels,refresh_kernels", GROWTH, ids=[g[0] for g in GROWTH])
def test_refresh_across_alphabet_growth(child, case, a0, a1, old_kernels, refresh_kernels):
    child(_refresh_across_alphabet_growth, case, a0, a1, old_kernels, refresh_kernels)


def _refresh_across_alphabet_growth(ctx, case, a0, a1, old_kernels, refresh_kernels):
    i = [g[0] for g in GROWTH].index(case)
    rng = np.random.default_rng(700 + i)
    off, act, ts = gen.make_log(2000, 0, 50, a0, seed=710 + i)
    log = ctx.load_log(off, act, ts, a0)
    old, names_old = _kernel_names(lambda: log.declare_counts(40))
    for k in old_kernels:
        assert _uses(names_old, k.replace("true", "false")), sorted(names_old)
    d = with_new(rng, off, ts, 25, 500, 10, a1)   # the batch uses the new activities
    new = _append(log, d, a1)
    got, names = _kernel_names(lambda: new.declare_counts_refresh(log, old, d.trace_idx))
    want = new.declare_counts(40)
    _same(got, want)
    assert got.tot[a0:].sum() > 0
    for k in refresh_kernels + [MERGE]:
        assert _uses(names, k), (k, sorted(names))
    assert not _uses(names, FULL)
    new.close()
    log.close()


def test_ids_outside_the_old_alphabet_that_the_new_one_covers_fall_back_to_a_full_count(child):
    child(_ids_outside_the_old_alphabet_that_the_new_one_covers_fall_back_to_a_full_count)


def _ids_outside_the_old_alphabet_that_the_new_one_covers_fall_back_to_a_full_count(ctx):
    rng = np.random.default_rng(9)
    off, act, ts = gen.make_log(2000, 0, 40, 14, seed=10)   # ids 0..13 on an alphabet of 10: act_valid is false
    d = with_new(rng, off, ts, 10, 300, 6, 14)
    got, want, names, old = _refresh(ctx, off, act, ts, 10, d, n_act_new=14)
    _same(got, want)
    assert _uses(names, FULL) and not _uses(names, MERGE), sorted(names)


def test_ids_outside_the_alphabet_that_it_does_not_cover_take_the_refresh_path(child):
    child(_ids_outside_the_alphabet_that_it_does_not_cover_take_the_refresh_path)


def _ids_outside_the_alphabet_that_it_does_not_cover_take_the_refresh_path(ctx):
    rng = np.random.default_rng(11)
    off, act, ts = gen.make_log(2000, 0, 40, 14, seed=12)   # ids 10..13 stay outside an alphabet of 10
    d = with_new(rng, off, ts, 10, 300, 6, 10, act_hi=14)
    got, want, names, _ = _refresh(ctx, off, act, ts, 10, d)
    _same(got, want)
    assert _uses(names, MERGE) and not _uses(names, FULL), sorted(names)


# ------------------------------------------------------------------------------------------------ histogram edges
def _repeat_log(n_traces, n_act, reps, seed):
    """Traces of `reps` occurrences of activity 0 among random others (timestamps ascending)."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(reps, reps + 8, size=n_traces)
    off = np.zeros(n_traces + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    act = np.zeros(int(off[-1]), dtype=np.int32)
    for t in range(n_traces):
        row = rng.integers(1, n_act, size=int(lens[t])).astype(np.int32)
        row[rng.choice(int(lens[t]), size=reps, replace=False)] = 0
        act[off[t]:off[t + 1]] = row
    ts = gen.T0_MS + np.arange(len(act), dtype=np.int64) * 1000
    return off, act, ts


HIST = [("k_cap_1", 1, 3, None), ("k_cap_40", 40, 3, None), ("cross_hs", 40, HS - 2, None), ("cross_hs_serial", 40, HS - 2, "SIESTA_K3_SERIAL"),
        ("cross_hs_any", 40, HS - 2, "SIESTA_K3_ANY"), ("to_overflow", 20, 20, None), ("to_overflow_serial", 20, 20, "SIESTA_K3_SERIAL"),
        ("to_overflow_any", 20, 20, "SIESTA_K3_ANY")]


@pytest.mark.parametrize("case,k_cap,reps,env", HIST, ids=[h[0] for h in HIST])
def test_histogram_edges(child, case, k_cap, reps, env):
    child(_histogram_edges, case, k_cap, reps, env, env=env)


def _histogram_edges(ctx, case, k_cap, reps, env):
    """An activity's count in a trace moves across HS (shared-memory buckets -> direct global atomics) or from k_cap to
    k_cap + 1 (hist -> hist_overflow)."""
    i = [h[0] for h in HIST].index(case)
    off, act, ts = _repeat_log(800, 6, reps, 800 + i)
    T = len(off) - 1
    listed = np.arange(0, T, 3, dtype=np.int64)
    b_off = np.arange(len(listed) + 1, dtype=np.int64) * 3
    b_act = np.zeros(int(b_off[-1]), dtype=np.int32)   # three more of activity 0
    b_ts = np.repeat(ts[off[listed + 1] - 1], 3) + np.tile([1000, 2000, 3000], len(listed))
    d = ingest.SeqDelta(listed, b_off, b_act, b_ts, 0, 6)
    got, want, names, old = _refresh(ctx, off, act, ts, 6, d, k_cap=k_cap)
    _same(got, want)
    assert _uses(names, MERGE)
    if case.startswith("to_overflow"):
        assert got.hist_overflow > old.hist_overflow and got.hist[0, k_cap] < old.hist[0, k_cap]
    if case.startswith("cross_hs"):
        assert got.hist[0, HS:].sum() > 0 and old.hist[0, HS:].sum() == 0


# ------------------------------------------------------------------------------------------------ scale and chaining
@pytest.mark.parametrize("env", [None, "SIESTA_K3_ANY"])
def test_more_listed_traces_than_a_launch_holds_at_once(child, env):
    child(_more_listed_traces_than_a_launch_holds_at_once, env, env=env)


def _more_listed_traces_than_a_launch_holds_at_once(ctx, env):
    """300 000 traces, 270 000 listed: every CTA of the pair kernel takes several batches of 32 traces, and the any kernel
    more rows than its grid cap of two CTAs per SM."""
    rng = np.random.default_rng(21)
    off, act, ts = gen.make_log(300_000, 0, 12, 10, seed=22)
    d = with_new(rng, off, ts, 2000, 268_000, 4, 10)
    assert len(d.trace_idx) > 262_144
    got, want, names, _ = _refresh(ctx, off, act, ts, 10, d)
    _same(got, want)
    assert _uses(names, ANY_WL if env else PAIRS_WL.format(2)) and _uses(names, MERGE), sorted(names)


def test_three_chained_refreshes_equal_a_full_count(child):
    child(_three_chained_refreshes_equal_a_full_count)


def _three_chained_refreshes_equal_a_full_count(ctx):
    rng = np.random.default_rng(31)
    off, act, ts = gen.make_log(3000, 0, 30, 12, seed=32)
    logs = [ctx.load_log(off, act, ts, 12)]
    cols = (off, act, ts)
    counts = [logs[0].declare_counts(40)]
    first = counts[0].packed.copy()
    union = np.zeros(0, dtype=np.int64)
    for step, n_act in enumerate((12, 14, 14)):
        d = with_new(rng, cols[0], cols[2], 50, 400, 6, n_act)
        cols = ingest.merge_delta(*cols, d)
        logs.append(_append(logs[-1], d, n_act))
        counts.append(logs[-1].declare_counts_refresh(logs[-2], counts[-1], d.trace_idx))
        union = np.union1d(union, d.trace_idx)
    want = logs[-1].declare_counts(40)
    _same(counts[-1], want)
    assert np.array_equal(want.packed, ctx.load_log(*cols, 14).declare_counts(40).packed)
    # one refresh over the whole chain with the union of the lists
    got, names = _kernel_names(lambda: logs[-1].declare_counts_refresh(logs[0], counts[0], union))
    _same(got, want)
    assert _uses(names, MERGE)
    assert np.array_equal(logs[0].declare_counts(40).packed, first)
    for lg in logs:
        lg.close()


# ------------------------------------------------------------------------------------------------ other entry points
def test_device_variant_with_caller_tensors_and_a_stream(child):
    child(_device_variant_with_caller_tensors_and_a_stream)


def _device_variant_with_caller_tensors_and_a_stream(ctx):
    import torch
    rng = np.random.default_rng(41)
    off, act, ts = gen.make_log(2000, 0, 40, 12, seed=42)
    log = ctx.load_log(off, act, ts, 12)
    old = log.declare_counts(40)
    for n_act in (12, 15):
        d = with_new(rng, off, ts, 20, 400, 6, n_act)
        new = _append(log, d, n_act)
        want = new.declare_counts(40)
        stream = torch.cuda.Stream(device=0)
        d_old = torch.from_numpy(old.packed.copy()).cuda(0)
        d_out = d_old if n_act == 12 else torch.full((len(want.packed),), -7, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()   # the tensors are filled on torch's stream, the refresh runs on `stream`
        ms, names = _kernel_names(lambda: new.declare_counts_refresh_device(log, d_old, d_out, d.trace_idx, 40,
                                                                            stream=stream.cuda_stream))
        stream.synchronize()
        assert ms >= 0 and _uses(names, MERGE)
        assert np.array_equal(d_out.cpu().numpy(), want.packed), n_act
        new.close()
    log.close()


def test_multi_log_refresh_equals_the_multi_count(child):
    child(_multi_log_refresh_equals_the_multi_count)


def _multi_log_refresh_equals_the_multi_count(ctx):
    from sequencedetectionqueryexecutor_b200 import api
    rng = np.random.default_rng(51)
    off, act, ts = gen.make_log(4000, 0, 40, 16, seed=52)
    with api.Multi([0, 0]) as m:
        ml = m.load_log(off, act, ts, 16)
        old = ml.declare_counts(40)
        d = with_new(rng, off, ts, 60, 1200, 6, 18)
        ml2 = ml.append(d.trace_idx, d.batch_off, d.act, d.ts_ms, d.n_new_traces, 18)
        got, names = _kernel_names(lambda: ml2.declare_counts_refresh(ml, old, d.trace_idx))
        want = ml2.declare_counts(40)
        _same(got, want)
        assert _uses(names, MERGE) and _uses(names, PAIRS_WL.format(2)) and not _uses(names, FULL), sorted(names)
        with pytest.raises(ValueError):
            ml2.declare_counts_refresh(ml2, old, d.trace_idx)   # counts of 16 activities for a log of 18
        ml2.close()
        ml.close()


def test_declare_miner_gives_the_same_templates_on_refreshed_counts(child):
    child(_declare_miner_gives_the_same_templates_on_refreshed_counts)


def _declare_miner_gives_the_same_templates_on_refreshed_counts(ctx):
    from sequencedetectionqueryexecutor_b200.declare import DeclareMiner
    rng = np.random.default_rng(61)
    off, act, ts = gen.make_log(3000, 1, 30, 8, seed=62)
    d = with_new(rng, off, ts, 100, 800, 6, 8)
    got, want, _, _ = _refresh(ctx, off, act, ts, 8, d)
    names = [f"a{i}" for i in range(8)]
    T = len(off) - 1 + d.n_new_traces
    a, b = DeclareMiner(got, names, T), DeclareMiner(want, names, T)
    modes = ["existence", "absence", "exactly", "co-existence", "choice", "exclusive-choice", "responded-existence"]
    assert a.existences(modes, 0.2) == b.existences(modes, 0.2)
    assert a.positions("both", 0.05) == b.positions("both", 0.05)
    for mode in ("simple", "alternate", "chain"):
        assert a.ordered_relations(mode, "succession", 0.1) == b.ordered_relations(mode, "succession", 0.1)


# ------------------------------------------------------------------------------------------------ refused calls
SENTINEL = -0x5EED


def _raw(old_log, new_log, trace_idx, k_cap, old_packed, n_out, n_listed=None):
    """siesta_declare_counts_refresh through ctypes -> (rc, out) with out pre-filled with a sentinel."""
    from sequencedetectionqueryexecutor_b200._lib import lib
    out = np.full(max(n_out, 1), SENTINEL, dtype=np.int64)
    ti = None if trace_idx is None else np.ascontiguousarray(trace_idx, dtype=np.int64)
    n = (0 if ti is None else len(ti)) if n_listed is None else n_listed
    rc = lib().siesta_declare_counts_refresh(old_log._h if old_log else None, new_log._h if new_log else None,
                                             C.c_void_p(ti.ctypes.data) if ti is not None and len(ti) else None, n, k_cap,
                                             C.c_void_p(old_packed.ctypes.data), C.c_void_p(out.ctypes.data), None)
    return rc, out


def test_refused_calls_leave_out_untouched(child):
    child(_refused_calls_leave_out_untouched)


def _refused_calls_leave_out_untouched(ctx):
    from sequencedetectionqueryexecutor_b200 import api
    rng = np.random.default_rng(71)
    off, act, ts = gen.make_log(1500, 1, 30, 10, seed=72)
    T = len(off) - 1
    log = ctx.load_log(off, act, ts, 10)
    old = log.declare_counts(40)
    d = with_new(rng, off, ts, 20, 300, 6, 10, min_len=1)
    new = _append(log, d)
    n_out = len(new.declare_counts(40).packed)
    ti = d.trace_idx
    touched = ti[ti < T]
    cases = {
        "null_log": (None, new, ti, 40),
        "null_trace_idx": (log, new, None, 40, len(ti)),
        "k_cap_0": (log, new, ti, 0),
        "not_ascending": (log, new, ti[::-1], 40),
        "outside": (log, new, np.append(ti, new.n_traces), 40),
        "new_trace_missing": (log, new, ti[:-1], 40),
        "unlisted_length_changed": (log, new, np.delete(ti, 3), 40),
        "fewer_traces": (new, log, touched, 40),
    }
    for name, args in cases.items():
        rc, out = _raw(*args[:4], old.packed, n_out, *args[4:])
        assert rc == abi.E_INVALID and (out == SENTINEL).all(), name
    # smaller alphabet: a batch that adds no trace, on a larger dictionary, refreshed the wrong way round
    d2 = with_new(rng, off, ts, 0, 100, 4, 10)
    grown = _append(log, d2, 12)
    rc, out = _raw(grown, log, d2.trace_idx, 40, grown.declare_counts(40).packed, n_out)
    assert rc == abi.E_INVALID and (out == SENTINEL).all()
    # derived and block-cyclic logs
    derived = log.filter_time(None, None)
    rc, out = _raw(derived, new, ti, 40, old.packed, n_out)
    assert rc == abi.E_INVALID and (out == SENTINEL).all()
    blocked = ctx.load_log(off, act, ts, 10)
    blocked.set_blocks([0, T], [0])
    rc, out = _raw(blocked, new, ti, 40, old.packed, n_out)
    assert rc == abi.E_INVALID and (out == SENTINEL).all()
    # another context
    with api.Context(0) as other:
        far = other.load_log(*ingest.merge_delta(off, act, ts, d), 10)
        rc, out = _raw(log, far, ti, 40, old.packed, n_out)
        assert rc == abi.E_INVALID and (out == SENTINEL).all()
        far.close()
    # an alphabet above 4096
    huge = _append(log, d, 4097)
    rc, out = _raw(log, huge, ti, 40, old.packed, 8)
    assert rc == abi.E_UNSUPPORTED and (out == SENTINEL).all()
    # counts of another alphabet
    with pytest.raises(ValueError):
        new.declare_counts_refresh(grown, old, d2.trace_idx)
    for lg in (huge, blocked, derived, grown, new, log):
        lg.close()
