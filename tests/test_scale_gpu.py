"""Kernels at sizes where their multi-level and looping parts run, against the CPU oracle and the host restatements.

- The placement of /detection (detect.cu) scans per-block sums of 256 candidates in chunks of 1 024 blocks; the second
  level (the `top` term of gather_kernel / gather_uniform_kernel) only exists past 262 144 candidates.
- row_scan_kernel (intersect.cu) scans 1 024 block counts per pass and carries the total into the next pass: every
  posting list, intersection and candidate list past 262 144 traces goes through that carry.
- pair_stats_kernel, pair_flags_kernel, the log-view kernels, the declare kernels and the explore kernels are
  grid-stride loops: a warp (or CTA) handles a second trace only when the log has more traces than the capped grid.

Every test asserts from the device's SM count and the launchers' constants that it reaches the part it is about."""
import os

import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200 import ingest
from tests import gen

pytestmark = pytest.mark.gpu

N_, P_, S_, X_, O_ = abi.STATE_NORMAL, abi.STATE_KLEENE_PLUS, abi.STATE_KLEENE_STAR, abi.STATE_NEGATIVE, abi.STATE_OR
GT = 256              # candidates per placement block (detect.cu)
SC = 1024             # blocks per chunk of the placement's first-level scan (detect.cu) and per pass of row_scan_kernel
IT = 256              # flags per block of the compaction (intersect.cu)
WARPS_PER_SM = 64     # resident warps an SM holds at most
THREADS = max(1, min(32, os.cpu_count() or 1))   # oracle threads


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _launches():
    from sequencedetectionqueryexecutor_b200 import api
    return api.kernel_launches()


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ placement
@pytest.fixture(scope="module")
def big_log(ctx):
    """300 000 short traces, then 400 traces of 120 - 200 events over the first three activities (beyond the mask
    kernels' 64 relevant events: class NK answers them on K1-L), all in the second scan chunk."""
    off, act, ts = gen.make_log(300_000, 0, 30, 6, seed=0xB16, max_gap_s=300, jitter_ms=True)
    l_off, l_act, l_ts = gen.make_log(400, 120, 200, 3, seed=0xB17, max_gap_s=60)
    off = np.concatenate([off, off[-1] + l_off[1:]])
    act = np.concatenate([act, l_act])
    ts = np.concatenate([ts, l_ts])
    log = ctx.load_log(off, act, ts, 6)
    yield off, act, ts, log
    log.close()


PLACEMENT_CASES = [
    # (name, states, flags, env) - uniform gather: class NK, first-largest, three events per occurrence
    ("uniform gather", [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])], 0, None),
    ("general gather for a uniform result", [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])], 0,
     "SIESTA_NO_UNIFORM_GATHER"),
    ("returnAll", [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL, None),
    ("returnAll negative", [dict(kind=N_, types=[0]), dict(kind=X_, types=[3]), dict(kind=N_, types=[1])],
     abi.F_RETURN_ALL | abi.F_EVT_POS, None),
    ("NP1 closed form", [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], 0, None),
    ("run-list engine", [dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])],
     abi.F_RETURN_ALL, None),
]


@pytest.mark.parametrize("name,states,flags,env", PLACEMENT_CASES, ids=[c[0] for c in PLACEMENT_CASES])
def test_placement_past_one_scan_chunk_equals_the_oracle(big_log, monkeypatch, name, states, flags, env):
    off, act, ts, log = big_log
    n_cand = len(off) - 1
    assert n_cand > SC * GT, "fewer candidates than one chunk of the placement's scan"
    if env:
        monkeypatch.setenv(env, "1")
    nfa = abi.make_nfa(states)
    got = log.detect(nfa, flags=flags)
    want = oracle.detect(off, act, ts, nfa, flags=flags, n_threads=THREADS)
    if got.n_unsupported:   # the Kleene shapes list long traces (beyond the engine's limits); every other trace is exact
        out = set(got.unsupported_trace_idx.tolist())
        assert any(s["kind"] in (P_, S_) for s in states) and out <= set(range(300_000, n_cand)), name
        assert got.as_dict() == {t: o for t, o in want.as_dict().items() if t not in out}, name
    else:
        ok, why = got.same_as(want)
        assert ok, (name, why)
    assert want.n_traces > 0 and want.trace_idx[-1] >= SC * GT, "no match in the second chunk"


def test_placement_with_candidates_and_device_result(big_log):
    """A candidate list past one chunk, and detect_device(...).tensors() equal to the host-buffer result."""
    off, act, ts, log = big_log
    rng = np.random.default_rng(3)
    cand = np.sort(rng.choice(len(off) - 1, size=280_000, replace=False)).astype(np.int64)
    assert len(cand) > SC * GT
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 4]), dict(kind=N_, types=[2])])
    host = log.detect(nfa, cand=cand, flags=abi.F_RETURN_ALL)
    ok, why = host.same_as(oracle.detect(off, act, ts, nfa, cand=cand, flags=abi.F_RETURN_ALL, n_threads=THREADS))
    assert ok, why
    import torch
    d_cand = torch.from_numpy(cand).cuda()
    dm = log.detect_device(nfa, d_cand=d_cand, flags=abi.F_RETURN_ALL)
    try:
        t = dm.tensors(0)
        torch.cuda.synchronize()
        for k in ("trace_idx", "occ_off", "ev_off", "ev_pos", "ev_rank", "ev_act", "ev_ts_ms", "err_trace_idx"):
            assert np.array_equal(t[k].cpu().numpy(), getattr(host, k)), k
    finally:
        dm.close()


def test_class_nk_long_traces_stage_on_k1l_past_one_chunk(big_log, monkeypatch):
    """Class NK with traces beyond 64 relevant events: K1-L answers them and stages in its own region, behind K1-P's and
    the staged kernels'.  Without K1-L (SIESTA_K1_NO_LONG) one kernel fewer runs and exactly those traces are listed."""
    off, act, ts, log = big_log
    lens = np.diff(off)
    long_traces = np.nonzero(lens > 64)[0]
    assert len(long_traces) == 400 and long_traces[0] >= SC * GT
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])])
    for flags in (0, abi.F_RETURN_ALL, abi.F_COUNT_MATCHES):
        want = oracle.detect(off, act, ts, nfa, flags=flags, n_threads=THREADS)
        n0 = _launches()
        got = log.detect(nfa, flags=flags)
        n_long = _launches() - n0
        assert got.n_unsupported == 0
        ok, why = got.same_as(want)
        assert ok, (flags, why)
        assert set(long_traces.tolist()) & set(got.trace_idx.tolist()), "no long trace matches"
        monkeypatch.setenv("SIESTA_K1_NO_LONG", "1")
        n0 = _launches()
        got2 = log.detect(nfa, flags=flags)
        n_plain = _launches() - n0
        monkeypatch.delenv("SIESTA_K1_NO_LONG")
        assert n_long != n_plain
        out = set(got2.unsupported_trace_idx.tolist())
        assert out and out <= set(long_traces.tolist())
        assert got2.as_dict() == {t: o for t, o in want.as_dict().items() if t not in out}


# ------------------------------------------------------------------------------------------------ pair index
def test_index_intersection_and_candidates_past_one_scan_pass(ctx):
    """build_index with 32 pairs (the most one call takes), (a, a) pairs and a pair naming an activity outside the
    alphabet, on more traces than one pass of row_scan_kernel and than pair_flags_kernel's grid has warps."""
    n_act = 34
    off, act, ts = gen.make_log(300_011, 10, 40, n_act, seed=0x1D3, max_gap_s=60)
    T = len(off) - 1
    assert (T + IT - 1) // IT > SC, "one pass of row_scan_kernel covers the log"
    assert T / (_sms() * 8 * (IT // 32)) >= 2, "pair_flags_kernel's warps handle one trace each"
    pairs = [(a, (a + 1) % 30) for a in range(24)] + [(0, 0), (5, 5), (29, 29), (30, 31), (31, 30), (32, 33), (33, 0),
                                                       (1, n_act + 3)]
    assert len(pairs) == 32
    log = ctx.load_log(off, act, ts, n_act)
    try:
        idx = log.build_index(pairs)
        lists = [oracle.posting_list(off, act, a, b) for a, b in pairs]
        for i, (a, b) in enumerate(pairs):
            assert np.array_equal(idx.posting_list(i), lists[i]), (a, b)
        assert len(lists[-1]) == 0 and all(len(x) and x[-1] >= SC * IT for x in lists[:-1])
        sels = [[3], [0, 1], [24, 25], [2, 2], [4, 4, 9], list(range(31)), list(range(32))]
        wants = [oracle.intersect([lists[i] for i in sorted(set(s))]) for s in sels]
        assert len(wants[1]) and wants[1][-1] >= SC * IT
        for s, w in zip(sels, wants):
            assert np.array_equal(idx.intersect(s), w), s
        exps = [[0, 1], [24], [2, 3, 4], [31], [26, 27, 28, 29]]
        want_c = np.zeros(0, dtype=np.int64)
        for x in exps:
            want_c = np.union1d(want_c, oracle.intersect([lists[i] for i in x]))
        assert np.array_equal(idx.candidates(exps), want_c)
        idx.close()
        # the same lists supplied by the caller
        idx2 = log.load_index(pairs, lists)
        for s, w in zip(sels, wants):
            assert np.array_equal(idx2.intersect(s), w), s
        assert np.array_equal(idx2.candidates(exps), want_c)
        idx2.close()
    finally:
        log.close()


# ------------------------------------------------------------------------------------------------ counting and views
def test_pair_stats_where_warps_loop(ctx):
    """Kernel K4 with 81 pairs (three passes of 32) on more traces than twice the resident warps."""
    off, act, ts = gen.make_log(40_000, 0, 60, 9, seed=0x57A7, max_gap_s=900, jitter_ms=True)
    assert (len(off) - 1) / (_sms() * WARPS_PER_SM) >= 2
    every = [(a, b) for a in range(9) for b in range(9)]
    log = ctx.load_log(off, act, ts, 9)
    try:
        got, _ = log.pair_stats(every)
    finally:
        log.close()
    assert got == oracle.pair_stats(off, act, ts, every)


@pytest.mark.parametrize("max_len", [64, 100])
def test_declare_counts_where_ctas_loop(ctx, monkeypatch, max_len):
    """Kernel K3 on its three paths: position masks (<= 32 activities, <= 64 and <= 128 events), the serial kernels
    (SIESTA_K3_SERIAL) and the any-alphabet kernel (SIESTA_K3_ANY), each on more work than its grid holds at once."""
    A, T = 20, 100_000
    off, act, ts = gen.make_log(T, 0, max_len, A, seed=0xDEC + max_len, zipf=1.1)
    assert int(np.diff(off).max()) <= 128 and A <= 32, "the log leaves the position-mask kernel"
    n_pairs = A * (A - 1) // 2
    threads = max(32, min(256, (n_pairs + 31) // 32 * 32))     # siesta_declare_counts_device, one pair per thread
    per_sm = min(32, WARPS_PER_SM // (threads // 32))
    assert (T + 31) // 32 >= 2 * _sms() * per_sm, "the pair kernel's CTAs take one batch each"
    assert T / (_sms() * WARPS_PER_SM) >= 2
    want = oracle.declare_counts(off, act, A, 40)
    log = ctx.load_log(off, act, ts, A)
    try:
        log.declare_counts(k_cap=40)   # the first call measures the longest trace
        launches = {}
        for knob in (None, "SIESTA_K3_SERIAL", "SIESTA_K3_ANY"):
            if knob:
                monkeypatch.setenv(knob, "1")
            n0 = _launches()
            got = log.declare_counts(k_cap=40)
            launches[knob] = _launches() - n0
            if knob:
                monkeypatch.delenv(knob)
            assert np.array_equal(got.packed, want.packed), knob
    finally:
        log.close()
    assert launches[None] != launches["SIESTA_K3_SERIAL"], launches


def test_filter_time_where_warps_loop(ctx):
    """lv_count_kept_kernel / lv_copy_kept_kernel on more traces than twice their capped grid's warps, then /detection on
    the view against the oracle on the restated window."""
    off, act, ts = gen.make_log(60_000, 0, 40, 8, seed=0xF17, max_gap_s=400, jitter_ms=True)
    T = len(off) - 1
    assert T / (_sms() * 16 * 8) >= 2, "every warp of the log-view grid handles one trace"
    lo, hi = int(ts.min()), int(ts.max())
    frm, til = lo + (hi - lo) // 5, lo + (hi - lo) * 3 // 4
    w_off, w_act, w_ts, kept = ingest.filter_time_range(off, act, ts, frm, til)
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 900)]),
                        dict(kind=X_, types=[3]), dict(kind=N_, types=[4])])
    log = ctx.load_log(off, act, ts, 8)
    try:
        view = log.filter_time(frm, til)
        assert (view.n_traces, view.n_events) == (T, len(w_act))
        assert np.array_equal(view.source_events(), kept)
        for flags in (0, abi.F_RETURN_ALL):
            ok, why = view.detect(nfa, flags=flags).same_as(oracle.detect(w_off, w_act, w_ts, nfa, flags=flags, n_threads=THREADS))
            assert ok, (flags, why)
        view.close()
    finally:
        log.close()


def test_group_where_warps_loop(ctx):
    """The group kernels (one warp per group) on more groups than twice their capped grid's warps, against the
    restatement of querySingleTableGroups, then /detection on the group streams."""
    from tests.test_logview_gpu import _java_groups
    off, act, ts = gen.make_log(60_000, 0, 8, 5, seed=0x6A0, max_gap_s=50)
    ts = (ts // 20000) * 20000   # equal timestamps across traces
    rng = np.random.default_rng(11)
    n_groups = 2 * _sms() * 16 * 8 + 101
    sizes = rng.integers(0, 4, size=n_groups)
    groups = [[int(x) for x in rng.choice(60_000, size=int(k), replace=True)] for k in sizes]
    types = [0, 1, 2]
    w_off, w_act, w_ts, w_src, ids = _java_groups(off, act, ts, groups, types)
    assert len(ids) > 1000
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])])
    log = ctx.load_log(off, act, ts, 5)
    try:
        glog, gids = log.group(groups, types)
        assert gids.tolist() == ids
        assert np.array_equal(glog.source_events(), w_src)
        for flags in (0, abi.F_RETURN_ALL):
            ok, why = glog.detect(nfa, flags=flags).same_as(oracle.detect(w_off, w_act, w_ts, nfa, flags=flags, n_threads=THREADS))
            assert ok, (flags, why)
        glog.close()
    finally:
        log.close()


def test_explore_accurate_past_the_grid_cap(ctx):
    """siesta_explore_accurate on more traces than its grid (sm_count * 8 CTAs of 8 warps, 4 traces in flight per warp)
    covers at once: completions and summed durations equal per-candidate oracle detection."""
    EX_BATCH = 4
    n_act = 8
    off, act, ts = gen.make_log(100_003, 0, 70, n_act, seed=0xE4, jitter_ms=True, max_gap_s=30)
    T = len(off) - 1
    cap = _sms() * 8
    assert (T + 8 * EX_BATCH - 1) // (8 * EX_BATCH) >= 2 * cap, "explore_prefix_kernel's grid is not capped"
    log = ctx.load_log(off, act, ts, n_act)
    try:
        for pat, fl in (([0, 1], 0), ([2], abi.F_EVT_POS)):
            comp, dur, _ = log.explore_accurate(pat, list(range(n_act)), fl)
            for c in range(n_act):
                nfa = abi.make_nfa([dict(kind=N_, types=[x]) for x in pat + [c]])
                want = oracle.detect(off, act, ts, nfa, flags=abi.F_RETURN_ALL | fl, n_threads=THREADS)
                s = want.ev_off
                d = int(np.sum(want.ev_ts_ms[s[1:] - 1] - want.ev_ts_ms[s[:-1]])) if want.n_occurrences else 0
                assert (comp[c], dur[c]) == (want.n_occurrences, d), (pat, fl, c)
    finally:
        log.close()
