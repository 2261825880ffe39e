"""Parity of the CUDA verification path (through the C-ABI) against the CPU oracle.  Bit-exact: matching
trace ids, reference-throw trace ids, selected occurrences and every output column."""
import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from tests import gen
from tests.kat import KATS, STREAM_TYPES

from sequencedetectionqueryexecutor_b200._lib import SiestaError

pytestmark = pytest.mark.gpu

N_, P_, S_, X_, O_ = abi.STATE_NORMAL, abi.STATE_KLEENE_PLUS, abi.STATE_KLEENE_STAR, abi.STATE_NEGATIVE, abi.STATE_OR


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


def _check(ctx, off, act, ts, n_act, states, flags, cand=None):
    nfa = abi.make_nfa(states)
    log = ctx.load_log(off, act, ts, n_act)
    try:
        got = log.detect(nfa, cand=cand, flags=flags)
    finally:
        log.close()
    want = oracle.detect(off, act, ts, nfa, cand=cand, flags=flags)
    if got.n_unsupported:   # traces beyond the engine's per-trace limits are listed, every other trace is exact
        out = set(got.unsupported_trace_idx.tolist())
        assert got.as_dict() == {t: o for t, o in want.as_dict().items() if t not in out}, f"states={states} flags={flags}"
        assert [t for t in got.err_trace_idx.tolist()] == [t for t in want.err_trace_idx.tolist() if t not in out]
        return got
    ok, why = got.same_as(want)
    assert ok, f"mismatch in {why}: states={states} flags={flags}"
    return got


@pytest.mark.parametrize("kat", KATS, ids=[k["name"] for k in KATS])
def test_reference_known_answer_tests(ctx, kat):
    """The reference's engine KATs (stream A B A C D A B E as EventPos), through the GPU path."""
    off = np.array([0, len(STREAM_TYPES)], dtype=np.int64)
    act = np.array(STREAM_TYPES, dtype=np.int32)
    ts = np.arange(len(STREAM_TYPES), dtype=np.int64) * 1000
    got = _check(ctx, off, act, ts, 5, kat["states"], abi.F_EVT_POS | abi.F_COUNT_MATCHES)
    assert got.n_matches_emitted == kat["expected"], kat["where"]
    if kat["matches"]:
        assert got.as_dict() == {0: [max(kat["matches"], key=len)]}
    else:
        assert got.n_traces == 0


@pytest.mark.parametrize("seed", range(4))
def test_random_nfas_all_kinds(ctx, seed):
    rng = np.random.default_rng(5000 + seed)
    n_ok = 0
    for it in range(60):
        n_act = int(rng.integers(3, 7))
        off, act, ts = gen.make_log(300, 0, 24, n_act, seed=int(rng.integers(1 << 30)), max_gap_s=300,
                                    jitter_ms=bool(rng.integers(0, 2)))
        states = gen.random_nfa(rng, n_act)
        flags = 0
        if rng.random() < 0.5:
            flags |= abi.F_EVT_POS
        if rng.random() < 0.5:
            flags |= abi.F_RETURN_ALL
        if rng.random() < 0.15:
            flags |= abi.F_ONLY_APPEARANCES
        if rng.random() < 0.25:
            flags |= abi.F_COUNT_MATCHES
        if rng.random() < 0.15:
            flags |= abi.F_LITERAL_RUNS
        try:
            got = _check(ctx, off, act, ts, n_act, states, flags)
        except SiestaError as e:  # beyond the engine's documented limits: reported, never silently wrong
            assert e.code == abi.E_UNSUPPORTED
            continue
        n_ok += got.n_ref_errors == 0
    assert n_ok > 20


@pytest.mark.parametrize("flags", [0, abi.F_RETURN_ALL, abi.F_EVT_POS, abi.F_EVT_POS | abi.F_RETURN_ALL])
def test_baseline_config_shapes(ctx, flags):
    # config 1: A_ B_ on 10k traces x ~40 events, 20 activities
    off, act, ts = gen.make_log(10_000, 30, 50, 20, seed=0x51E57A01)
    got = _check(ctx, off, act, ts, 20, [dict(kind=N_, types=[0]), dict(kind=N_, types=[1])], flags)
    assert got.n_traces > 1000
    # config 2 shape: a+ b* within 10 minutes
    off, act, ts = gen.make_log(4000, 100, 100, 20, seed=0x51E57A02, max_gap_s=120)
    st = [dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])]
    got = _check(ctx, off, act, ts, 20, st, flags)
    assert got.n_traces > 100
    # config 5 shape: a, (b|c), !d, e, f ; gap within 10 (0,1), gap atleast 2 (3,4)
    off, act, ts = gen.make_log(4000, 50, 50, 20, seed=0x51E57A05)
    st = [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
          dict(kind=X_, types=[3]), dict(kind=N_, types=[4]),
          dict(kind=N_, types=[5], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])]
    _check(ctx, off, act, ts, 20, st, flags)


def test_ragged_and_empty_inputs(ctx):
    # empty traces, traces with no relevant event, a single long trace, trace count not a multiple of the tile
    off, act, ts = gen.make_log(1001, 0, 3, 4, seed=9)
    _check(ctx, off, act, ts, 4, [dict(kind=N_, types=[0]), dict(kind=N_, types=[1])], 0)
    off, act, ts = gen.make_log(3, 700, 900, 50, seed=10)
    _check(ctx, off, act, ts, 50, [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL)
    # activity id unknown to the log and a log with zero events
    off, act, ts = gen.make_log(50, 5, 9, 4, seed=11)
    got = _check(ctx, off, act, ts, 4, [dict(kind=N_, types=[0]), dict(kind=N_, types=[17])], 0)
    assert got.n_traces == 0
    z = np.zeros(1, dtype=np.int64)
    got = _check(ctx, np.zeros(6, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int64), 4,
                 [dict(kind=N_, types=[0])], 0)
    assert got.n_traces == 0 and z[0] == 0


def test_candidate_lists(ctx):
    off, act, ts = gen.make_log(5000, 20, 40, 10, seed=12)
    rng = np.random.default_rng(3)
    cand = np.sort(rng.choice(5000, size=1777, replace=False)).astype(np.int64)
    st = [dict(kind=N_, types=[0]), dict(kind=X_, types=[3]), dict(kind=N_, types=[1])]
    got = _check(ctx, off, act, ts, 10, st, abi.F_RETURN_ALL, cand=cand)
    assert set(got.trace_idx.tolist()) <= set(cand.tolist())
    _check(ctx, off, act, ts, 10, st, 0, cand=np.zeros(0, dtype=np.int64))


def test_wide_engine_path(ctx):
    """Traces beyond the narrow configuration (32 relevant events / 64 live runs) re-run on the wide one."""
    off, act, ts = gen.make_log(500, 20, 45, 3, seed=77)
    _check(ctx, off, act, ts, 3, [dict(kind=P_, types=[0]), dict(kind=S_, types=[1])], 0)
    _check(ctx, off, act, ts, 3, [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL)


def test_limits_are_reported_not_silently_wrong(ctx):
    """A trace beyond the engine's per-trace limits does not fail the request (the reference has no limit,
    Engine.java:207-224): every other trace is answered exactly and the outliers are listed."""
    from sequencedetectionqueryexecutor_b200._lib import SiestaError
    off, act, ts = gen.make_log(300, 0, 40, 2, seed=5)
    long_off, long_act, long_ts = gen.make_log(3, 200, 200, 2, seed=6)          # ~200 relevant events per trace > 64
    # the three long traces go to positions 17, 18 and the very end
    cut = int(off[17])
    act2 = np.concatenate([act[:cut], long_act[:400], act[cut:], long_act[400:]])
    ts2 = np.concatenate([ts[:cut], long_ts[:400], ts[cut:], long_ts[400:]])
    lens = np.concatenate([np.diff(off)[:17], [200, 200], np.diff(off)[17:], [200]])
    off2 = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    outliers = [17, 18, len(lens) - 1]
    for states, flags, limited in (([dict(kind=N_, types=[0]), dict(kind=N_, types=[1])], 0, False),          # class NK: kernel K1-L answers them
                                   ([dict(kind=P_, types=[0]), dict(kind=S_, types=[1])], 0, True),
                                   ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[0])], abi.F_RETURN_ALL, True)):
        nfa = abi.make_nfa(states)
        log = ctx.load_log(off2, act2, ts2, 2)
        got = log.detect(nfa, flags=flags)
        log.close()
        want = oracle.detect(off2, act2, ts2, nfa, flags=flags)
        if not limited:
            assert got.n_unsupported == 0
            ok, why = got.same_as(want)
            assert ok, why
            continue
        assert got.unsupported_trace_idx.tolist() == outliers and got.n_unsupported == 3
        keep = ~np.isin(want.trace_idx, outliers)
        assert np.array_equal(got.trace_idx, want.trace_idx[keep])
        # the occurrences of the supported traces, one by one
        wd = want.as_dict()
        assert got.as_dict() == {t: o for t, o in wd.items() if t not in outliers}
    log = ctx.load_log(*gen.make_log(4, 5, 5, 2, seed=5), 2)
    with pytest.raises(SiestaError) as e:  # HEAD mode has no defined output when state 1 is kleeneClosure*
        log.detect(abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=S_, types=[1])]), flags=abi.F_MODE_HEAD)
    log.close()
    assert e.value.code == abi.E_UNSUPPORTED


def test_evaluate_events_and_sase_connector_mirror(ctx):
    """The reference-facing call shapes: SaseConnector.evaluate over host events, and the Python mirror."""
    from sequencedetectionqueryexecutor_b200 import sase
    off, act, ts = gen.make_log(2000, 30, 50, 20, seed=0x51E57A01, jitter_ms=True)
    names = [f"act{i:02d}" for i in range(20)]
    acts = sase.ActivityDictionary(names)
    pattern = sase.ComplexPattern([sase.EventSymbol("ACT00", 0, "_"), sase.EventSymbol("act01", 1, "||"),
                                   sase.EventSymbol("act02", 1, "_"), sase.EventSymbol("act03", 2, "!"),
                                   sase.EventSymbol("act04", 3, "_")],
                                  [sase.TimeConstraint(0, 1, 30, "within", "minutes")])
    nfa = pattern.getNfa(acts)
    want = oracle.detect(off, act, ts, nfa, flags=0)
    got = ctx.evaluate_events(off, act, ts, 20, nfa, flags=0)
    ok, why = got.same_as(want)
    assert ok, why
    log = ctx.load_log(off, act, ts, 20)
    occs = sase.SaseConnector(acts).evaluate(pattern, log, onlyAppearances=False)
    log.close()
    assert len(occs) == want.n_traces
    first = occs[0].occurrences[0].occurrence
    assert [e.name for e in first][0] == "act00" and first[0].timestamp_ms == want.ev_ts_ms[0]


def test_one_million_events_idempotent_and_sorted(ctx):
    """Size-independent properties at a size the oracle does not need to see: ascending trace ids, CSR offsets
    consistent, positions strictly increasing inside an occurrence, identical output on a second call."""
    off, act, ts = gen.make_log(20_000, 40, 60, 20, seed=99)
    log = ctx.load_log(off, act, ts, 20)
    st = [dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])]
    nfa = abi.make_nfa(st)
    a = log.detect(nfa, flags=abi.F_RETURN_ALL)
    b = log.detect(nfa, flags=abi.F_RETURN_ALL)
    log.close()
    assert a.same_as(b)[0]
    assert np.all(np.diff(a.trace_idx) > 0)
    assert a.occ_off[0] == 0 and a.occ_off[-1] == a.n_occurrences and a.ev_off[-1] == a.n_events
    lens = np.diff(a.ev_off)
    assert np.all(lens > 0)
    inner = np.ones(a.n_events, dtype=bool)
    inner[a.ev_off[:-1]] = False
    assert np.all(np.diff(a.ev_pos)[inner[1:]] > 0)


def test_device_result_views_and_single_rank_gather(ctx):
    """DeviceMatches.tensors(): zero-copy torch views of the HBM-resident result equal the host-buffer result."""
    import torch
    off, act, ts = gen.make_log(3000, 20, 40, 10, seed=21)
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])])
    log = ctx.load_log(off, act, ts, 10)
    host = log.detect(nfa, flags=abi.F_RETURN_ALL)
    dm = log.detect_device(nfa, flags=abi.F_RETURN_ALL)
    t = dm.tensors(0)
    torch.cuda.synchronize()
    for k in ("trace_idx", "occ_off", "ev_off", "ev_pos", "ev_rank", "ev_act", "ev_ts_ms"):
        assert np.array_equal(t[k].cpu().numpy(), getattr(host, k)), k
    dm.close()
    log.close()


def test_evaluate_events_streams_in_chunks(ctx, monkeypatch):
    """siesta_evaluate_events cuts the request into chunks of whole traces (copy of chunk c+1 overlaps the scan of
    chunk c) and rebases the chunk results on the device: the joined result must equal the oracle's, including the
    reference-throw list and empty / ragged traces at chunk borders."""
    monkeypatch.setenv("SIESTA_CHUNK_EVENTS", "3000")
    off, act, ts = gen.make_log(3000, 0, 60, 6, seed=31, jitter_ms=True)
    cases = [
        ([dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], 0),
        ([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2]), dict(kind=X_, types=[3]), dict(kind=N_, types=[4])], abi.F_RETURN_ALL),
        ([dict(kind=X_, types=[1]), dict(kind=P_, types=[2])], abi.F_EVT_POS),   # shape on which the Java engine throws
        ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_COUNT_MATCHES),
    ]
    for states, flags in cases:
        nfa = abi.make_nfa(states)
        want = oracle.detect(off, act, ts, nfa, flags=flags)
        got = ctx.evaluate_events(off, act, ts, 6, nfa, flags=flags)
        ok, why = got.same_as(want)
        assert ok, (why, states, flags)
    # one trace longer than the chunk budget, and a request without events
    off2, act2, ts2 = gen.make_log(3, 5000, 6000, 1000, seed=32)
    nfa = abi.make_nfa([dict(kind=N_, types=[0]), dict(kind=N_, types=[1])])
    assert ctx.evaluate_events(off2, act2, ts2, 1000, nfa).same_as(oracle.detect(off2, act2, ts2, nfa))[0]
    z = ctx.evaluate_events(np.zeros(4, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int64), 4, nfa)
    assert z.n_traces == 0 and z.occ_off.tolist() == [0]
    # offsets are validated chunk by chunk: a decreasing offset deep inside the request fails the call, nothing is read out of bounds
    bad = off.copy()
    bad[2000] = bad[1999] - 1
    with pytest.raises(SiestaError) as e:
        ctx.evaluate_events(bad, act, ts, 6, nfa)
    assert e.value.code == abi.E_INVALID


def test_evaluate_events_byte_activity_column(ctx, monkeypatch):
    """siesta_evaluate_events_act8: the activity column crosses the host link as one byte per event and is widened on the
    device chunk by chunk (chunks start at any event index, so the ragged ends of the 4-event groups are exercised);
    results equal the oracle's on the int32 column, with pinned (timestamps read in place) and pageable inputs."""
    import torch
    off, act, ts = gen.make_log(4000, 0, 70, 200, seed=77, max_gap_s=300, jitter_ms=True)
    act = (act % 7 + (act % 3 == 0) * 190).astype(np.int32)        # ids 0 .. 6 and 190 .. 196: both ends of the byte range
    act8 = act.astype(np.uint8)
    cases = [([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
               dict(kind=X_, types=[3]), dict(kind=N_, types=[190])], 0),
             ([dict(kind=P_, types=[0]), dict(kind=S_, types=[191], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], 0),
             ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL),
             ([dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[190])], abi.F_RETURN_ALL)]   # returnAll on K1-P
    p_off, p_act8, p_ts = (torch.from_numpy(x).pin_memory() for x in (off, act8, ts))
    for chunk in ("1000", "4099", None):
        if chunk:
            monkeypatch.setenv("SIESTA_CHUNK_EVENTS", chunk)
        else:
            monkeypatch.delenv("SIESTA_CHUNK_EVENTS")
        for states, flags in cases:
            nfa = abi.make_nfa(states)
            want = oracle.detect(off, act, ts, nfa, flags=flags)
            for a, b, c in ((off, act8, ts), (p_off.numpy(), p_act8.numpy(), p_ts.numpy())):
                got = ctx.evaluate_events(a, b, c, 200, nfa, flags=flags)
                ok, why = got.same_as(want)
                assert ok, (why, states, flags, chunk)
    with pytest.raises(SiestaError) as e:
        ctx.evaluate_events(off, act8, ts, 300, abi.make_nfa(cases[0][0]))     # 300 activities do not fit a byte
    assert e.value.code == abi.E_INVALID
    z = ctx.evaluate_events(np.zeros(4, dtype=np.int64), np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.int64), 4, abi.make_nfa(cases[0][0]))
    assert z.n_traces == 0


def test_filter_variants_long_traces_large_alphabets_bad_ids(ctx):
    """The filter of kernel K1 has three forms (<= 32 activities, <= 64, general) and two row widths; all must agree
    with the oracle.  Also: traces longer than 8192 events leave the narrow configuration, more than 7 pattern
    activities leave the class-plane filter, and activity ids outside [0, n_activities) never match."""
    N = N_
    for n_act, seed in ((20, 41), (50, 42), (300, 43)):
        off, act, ts = gen.make_log(1500, 10, 120, n_act, seed=seed, zipf=1.2 if n_act > 64 else None)
        b = 0 if n_act <= 64 else 9  # Zipf log: stay off the head of the distribution (<= 64 relevant events per trace)
        st = [dict(kind=N, types=[b]), dict(kind=O_, types=[b + 1, b + 2, b + 3]), dict(kind=X_, types=[b + 4]),
              dict(kind=N, types=[b + 5]), dict(kind=N, types=[b], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])]
        _check(ctx, off, act, ts, n_act, st, 0)
        _check(ctx, off, act, ts, n_act, [dict(kind=P_, types=[n_act - 1]), dict(kind=S_, types=[b])], abi.F_EVT_POS)
    # 9 pattern activities (> 7 classes)
    off, act, ts = gen.make_log(800, 20, 60, 12, seed=44)
    st = [dict(kind=O_, types=[0, 1, 2]), dict(kind=O_, types=[3, 4, 5]), dict(kind=O_, types=[6, 7, 8])]
    _check(ctx, off, act, ts, 12, st, abi.F_RETURN_ALL)
    # long traces: 9000-event traces with few relevant events
    off, act, ts = gen.make_log(6, 9000, 9500, 2000, seed=45)
    _check(ctx, off, act, ts, 2000, [dict(kind=N, types=[0]), dict(kind=N, types=[1])], 0)
    _check(ctx, off, act, ts, 2000, [dict(kind=P_, types=[3]), dict(kind=S_, types=[4])], 0)
    # ids outside the alphabet
    off, act, ts = gen.make_log(400, 10, 40, 8, seed=46)
    act = act.copy()
    act[::7] = -3
    act[3::11] = 8
    act[5::13] = 1 << 20
    _check(ctx, off, act, ts, 8, [dict(kind=N, types=[0]), dict(kind=N, types=[1])], 0)
    _check(ctx, off, act, ts, 8, [dict(kind=P_, types=[2]), dict(kind=S_, types=[3])], 0)


def test_pruning_then_verification_equals_verifying_everything(ctx):
    """Rows P1-P3 in front of V*: true pairs of the pattern (siesta_pattern_extract_pairs) -> posting lists of the
    resident log (siesta_index_build) -> union over the OR-expansions of the per-expansion intersections
    (siesta_candidates) -> siesta_detect(cand).  Under the SeqTable view a trace that lacks a true pair cannot match,
    so the pruned run must return exactly what the unpruned run and the oracle return."""
    from sequencedetectionqueryexecutor_b200 import sase
    off, act, ts = gen.make_log(6000, 5, 40, 12, seed=61)
    acts = sase.ActivityDictionary([f"act{i:02d}" for i in range(12)])
    patterns = [
        sase.ComplexPattern([sase.EventSymbol("act00", 0, "_"), sase.EventSymbol("act01", 1, "||"), sase.EventSymbol("act02", 1, "_"),
                             sase.EventSymbol("act03", 2, "!"), sase.EventSymbol("act04", 3, "_"), sase.EventSymbol("act05", 4, "_")],
                            [sase.GapConstraint(0, 1, 10, "within"), sase.GapConstraint(3, 4, 2, "atleast")]),
        sase.ComplexPattern([sase.EventSymbol("act00", 0, "_"), sase.EventSymbol("act01", 1, "+"), sase.EventSymbol("act02", 2, "*"),
                             sase.EventSymbol("act03", 3, "_")], []),
        sase.ComplexPattern([sase.EventSymbol("act06", 0, "_"), sase.EventSymbol("act07", 1, "_"), sase.EventSymbol("act06", 2, "_")], []),
    ]
    log = ctx.load_log(off, act, ts, 12)
    try:
        for p in patterns:
            cand = sase.pattern_candidates(p, log, acts)
            exps = p.extractPairsForPatternDetection(acts)
            want_c = np.zeros(0, dtype=np.int64)
            for x in exps:  # oracle: intersection per expansion, union over expansions
                want_c = np.union1d(want_c, oracle.intersect([oracle.posting_list(off, act, a, b) for a, b in x.truePairs]))
            assert np.array_equal(cand, want_c)
            assert 0 < len(cand) < 6000
            nfa = p.getNfa(acts)
            want = oracle.detect(off, act, ts, nfa, flags=abi.F_RETURN_ALL)
            pruned = log.detect(nfa, cand=cand, flags=abi.F_RETURN_ALL)
            ok, why = pruned.same_as(want)
            assert ok, why
    finally:
        log.close()


def test_explore_accurate_matches_per_candidate_detection(ctx):
    """Row X: siesta_explore_accurate = for every candidate, detection of pattern + candidate with
    clearOccurrences(true); completions and summed durations must equal what the oracle's detection gives."""
    from sequencedetectionqueryexecutor_b200 import sase
    n_act = 12
    off, act, ts = gen.make_log(5000, 10, 50, n_act, seed=81, jitter_ms=True)
    acts = sase.ActivityDictionary([f"act{i:02d}" for i in range(n_act)])
    base = [0, 1]
    log = ctx.load_log(off, act, ts, n_act)
    try:
        comp, dur, _ = log.explore_accurate(base, list(range(n_act)))
        for c in range(n_act):
            nfa = abi.make_nfa([dict(kind=N_, types=[x]) for x in base + [c]])
            want = oracle.detect(off, act, ts, nfa, flags=abi.F_RETURN_ALL)
            assert comp[c] == want.n_occurrences, c
            d = sum(int(want.ev_ts_ms[want.ev_off[o + 1] - 1] - want.ev_ts_ms[want.ev_off[o]]) for o in range(want.n_occurrences))
            assert dur[c] == d, c
        # shapes around the shared pass: traces beyond 64 events and more than 16 starts (overflow list -> general kernels),
        # the EventPos route, one- and three-event patterns, a candidate that repeats a pattern activity, unsorted timestamps
        for n_a, lens, pat, fl, shuffle in [(6, (40, 80), [0, 1], 0, False), (6, (0, 64), [2], abi.F_EVT_POS, False),
                                            (9, (20, 70), [0, 1, 2], 0, True), (4, (60, 64), [1, 1], abi.F_EVT_POS, False),
                                            (40, (50, 50), [0, 1, 2], 0, False)]:
            o2, a2, t2 = gen.make_log(3000, lens[0], lens[1], n_a, seed=83 + n_a, jitter_ms=True, max_gap_s=5)
            if shuffle:
                t2 = t2.copy()
                np.random.default_rng(5).shuffle(t2)
            l2 = ctx.load_log(o2, a2, t2, n_a)
            try:
                comp2, dur2, _ = l2.explore_accurate(pat, list(range(n_a)), fl)
            finally:
                l2.close()
            for c in range(n_a):
                nfa = abi.make_nfa([dict(kind=N_, types=[x]) for x in pat + [c]])
                want = oracle.detect(o2, a2, t2, nfa, flags=abi.F_RETURN_ALL | fl)
                d = sum(int(want.ev_ts_ms[want.ev_off[o + 1] - 1] - want.ev_ts_ms[want.ev_off[o]]) for o in range(want.n_occurrences))
                assert (comp2[c], dur2[c]) == (want.n_occurrences, d), (n_a, lens, pat, fl, c)
        props = sase.explore_accurate(["act00", "act01"], log, acts)
        assert [p.event for p in props] == [p.event for p in sorted(props, key=lambda p: (-p.completions / p.averageDuration, p.event))]
        assert {p.event for p in props} == {acts.names[c] for c in range(n_act) if comp[c] > 0}
        assert all(abs(p.averageDuration - dur[acts.id(p.event)] / 1000.0 / p.completions) < 1e-9 for p in props)
    finally:
        log.close()


def _block_layout(n_tr, n_occ, n_ev, n_err, n_unsup, all_cols):
    """Byte offsets of the result columns inside siesta_dev_matches.d_block, in the order include/siesta_gpu.h
    documents (each at a 256-byte aligned offset), and the block's size."""
    cols = [("trace_idx", n_tr * 8), ("occ_off", (n_tr + 1) * 8), ("ev_off", (n_occ + 1) * 8), ("ev_pos", n_ev * 4),
            ("err_trace_idx", n_err * 8)]
    if all_cols:
        cols += [("ev_rank", n_ev * 4), ("ev_act", n_ev * 4), ("ev_ts_ms", n_ev * 8)]
    cols.append(("unsupported_trace_idx", n_unsup * 8))
    off, o = {}, 0
    for name, nbytes in cols:
        off[name] = o
        o += (nbytes + 255) & ~255
    return off, o


def test_result_block_layout_and_shard_offsets(ctx):
    """The device result is one allocation with a documented layout, and a log marked as a shard returns global
    trace indices."""
    off, act, ts = gen.make_log(3000, 0, 40, 8, seed=91)
    nfa = abi.make_nfa([dict(kind=X_, types=[3]), dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])])
    want = oracle.detect(off, act, ts, nfa, flags=abi.F_RETURN_ALL)
    log = ctx.load_log(off, act, ts, 8)
    log.set_first_trace(1_000_000)
    dm = log.detect_device(nfa, flags=abi.F_RETURN_ALL)
    d = dm.dm
    assert (d.n_traces, d.n_occurrences, d.n_events, d.n_ref_errors) == (want.n_traces, want.n_occurrences, want.n_events, want.n_ref_errors)
    lay, total = _block_layout(d.n_traces, d.n_occurrences, d.n_events, d.n_ref_errors, d.n_unsupported, d.d_ev_rank)
    assert total == d.block_bytes
    for k, o in lay.items():
        assert getattr(d, "d_" + k) == d.d_block + o, k
    got = {k: v.cpu().numpy() for k, v in dm.tensors(0).items()}
    assert np.array_equal(got["trace_idx"], want.trace_idx + 1_000_000)
    assert np.array_equal(got["err_trace_idx"], want.err_trace_idx + 1_000_000)
    for k in ("occ_off", "ev_off", "ev_pos", "ev_rank", "ev_act", "ev_ts_ms"):
        assert np.array_equal(got[k], getattr(want, k)), k
    dm.close()
    log.close()


def test_concurrent_requests_on_one_log(ctx):
    """The reference serves concurrent requests (request-scoped plans on Tomcat threads): siesta_detect, siesta_evaluate_events
    and the counting calls on ONE log / ctx from several threads must each return their own exact result."""
    import threading
    off, act, ts = gen.make_log(20_000, 10, 60, 10, seed=101)
    log = ctx.load_log(off, act, ts, 10)
    jobs = [([dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 900)])], 0),
            ([dict(kind=N_, types=[2]), dict(kind=O_, types=[3, 4]), dict(kind=X_, types=[5]), dict(kind=N_, types=[6])], abi.F_RETURN_ALL),
            ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL),
            ([dict(kind=S_, types=[7]), dict(kind=N_, types=[8])], abi.F_EVT_POS)]
    wants = [oracle.detect(off, act, ts, abi.make_nfa(s), flags=f) for s, f in jobs]
    want_counts = oracle.declare_counts(off, act, 10, 40)
    errors = []

    def worker(i):
        try:
            s, f = jobs[i % len(jobs)]
            for rep in range(6):
                got = log.detect(abi.make_nfa(s), flags=f) if rep % 2 == 0 else ctx.evaluate_events(off, act, ts, 10, abi.make_nfa(s), flags=f)
                ok, why = got.same_as(wants[i % len(jobs)])
                if not ok:
                    errors.append((i, rep, why))
            if i == 0 and not np.array_equal(log.declare_counts(k_cap=40).packed, want_counts.packed):
                errors.append((i, "declare"))
        except Exception as e:  # noqa: BLE001
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    log.close()
    assert not errors, errors


@pytest.mark.parametrize("seed", range(3))
def test_raw_slot_kernel_nk_class(ctx, seed):
    """Kernel K1-P (class NK over raw position slots): random NK NFAs, trace lengths on both sides of the 64-slot
    limit (longer traces re-run on the staged kernel, > 24 relevant events on the wide one), alphabets of <= 32 and
    <= 64 activities, EventTs / EventPos routes, exact match counts, candidate lists."""
    from tests import soak_fast
    rng = np.random.default_rng(9100 + seed)
    n_match = 0
    for it in range(40):
        n_act = int(rng.choice([3, 5, 8, 20, 40, 64]))
        lo, hi = [(0, 30), (40, 70), (55, 66), (0, 130)][it % 4]
        off, act, ts = gen.make_log(700, lo, hi, n_act, seed=int(rng.integers(1 << 30)), max_gap_s=300)
        states = soak_fast.nk_nfa(rng, min(n_act, 8))
        for st in states:   # no time predicates on the EventTs route: those need relative seconds (staged kernel)
            st["preds"] = [p for p in st["preds"] if p[0] == abi.ATTR_POSITION or it % 2 == 0]
        flags = abi.F_EVT_POS if it % 2 == 0 else 0
        if rng.random() < 0.3:
            flags |= abi.F_COUNT_MATCHES
        if rng.random() < 0.2:
            flags |= abi.F_NO_EVENT_COLUMNS
        cand = None
        if rng.random() < 0.3:
            cand = np.sort(rng.choice(700, size=300, replace=False)).astype(np.int64)
        try:
            got = _check(ctx, off, act, ts, n_act, states, flags, cand=cand)
        except SiestaError as e:  # a trace with more than 64 relevant events: reported, never silently wrong
            assert e.code == abi.E_UNSUPPORTED
            continue
        n_match += got.n_traces
    assert n_match > 1000


def test_begin_finish_requests_in_flight(ctx):
    """siesta_detect_device_begin / _finish: several requests enqueued before any is finished, finished out of order,
    each equal to the oracle's result (and to the one-call form)."""
    off, act, ts = gen.make_log(6000, 10, 70, 10, seed=111)
    log = ctx.load_log(off, act, ts, 10)
    jobs = [([dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 900)])], 0),
            ([dict(kind=N_, types=[2]), dict(kind=O_, types=[3, 4]), dict(kind=X_, types=[5]), dict(kind=N_, types=[6])], 0),
            ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL),
            ([dict(kind=N_, types=[7]), dict(kind=N_, types=[8])], abi.F_EVT_POS | abi.F_COUNT_MATCHES)]
    try:
        pend = [log.detect_device_begin(abi.make_nfa(s), flags=f) for s, f in jobs]
        for i in (2, 0, 3, 1):
            dm = pend[i].finish()
            want = oracle.detect(off, act, ts, abi.make_nfa(jobs[i][0]), flags=jobs[i][1])
            assert (dm.n_traces, dm.n_occurrences, dm.n_events) == (want.n_traces, want.n_occurrences, want.n_events), i
            t = dm.tensors(0)
            assert np.array_equal(t["trace_idx"].cpu().numpy(), want.trace_idx) and np.array_equal(t["ev_pos"].cpu().numpy(), want.ev_pos), i
            assert np.array_equal(t["ev_ts_ms"].cpu().numpy(), want.ev_ts_ms) and np.array_equal(t["ev_off"].cpu().numpy(), want.ev_off), i
            dm.close()
        # a request that is begun and finished at once equals the one-call form
        a = log.detect_device_begin(abi.make_nfa(jobs[1][0]), flags=0).finish()
        b = log.detect_device(abi.make_nfa(jobs[1][0]), flags=0)
        assert (a.n_traces, a.n_events) == (b.n_traces, b.n_events)
        a.close()
        b.close()
    finally:
        log.close()


def test_wrapped_device_logs_are_validated(ctx):
    """siesta_log_wrap_device checks the caller's CSR on the device: offsets that decrease, do not start at 0 or do not end at
    n_events, and null columns, are refused instead of becoming out-of-bounds reads in every kernel."""
    import torch

    from sequencedetectionqueryexecutor_b200._lib import SiestaError
    off, act, ts = gen.make_log(50, 1, 9, 4, seed=1)
    d_act, d_ts = torch.from_numpy(act).cuda(), torch.from_numpy(ts).cuda()
    good = ctx.wrap_log(torch.from_numpy(off).cuda(), d_act, d_ts, 4)
    assert good.n_traces == 50
    good.close()
    for mutate in (lambda o: o.__setitem__(0, 1), lambda o: o.__setitem__(-1, o[-1] - 1), lambda o: o.__setitem__(10, o[12] + 1),
                   lambda o: o.__setitem__(5, -3)):
        bad = off.copy()
        mutate(bad)
        with pytest.raises(SiestaError) as e:
            ctx.wrap_log(torch.from_numpy(bad).cuda(), d_act, d_ts, 4)
        assert e.value.code == abi.E_INVALID


def test_evaluate_events_reads_pinned_timestamps_in_place(ctx):
    """Without a time constraint siesta_evaluate_events leaves a page-locked timestamp column on the host and the kernels
    read the reported events' timestamps through the mapping; results equal the oracle's either way."""
    import torch
    off, act, ts = gen.make_log(20000, 0, 60, 12, seed=404, max_gap_s=500, jitter_ms=True)
    p_off, p_act, p_ts = (torch.from_numpy(x).pin_memory() for x in (off, act, ts))
    cases = [([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
               dict(kind=X_, types=[3]), dict(kind=N_, types=[4])], 0),                         # K1-P
             ([dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], 0),  # staged kernel, run-list engine
             ([dict(kind=N_, types=[0]), dict(kind=N_, types=[1])], abi.F_EVT_POS),
             # returnAll on K1-P: the overlap test of the few traces with more than one engine match reads through the mapping as well
             ([dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
               dict(kind=X_, types=[3]), dict(kind=N_, types=[4])], abi.F_RETURN_ALL),
             ([dict(kind=N_, types=[0]), dict(kind=N_, types=[1])], abi.F_RETURN_ALL | abi.F_COUNT_MATCHES),
             ([dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], 0)]  # matches on time: copied
    for states, flags in cases:
        nfa = abi.make_nfa(states)
        want = oracle.detect(off, act, ts, nfa, flags=flags)
        got = ctx.evaluate_events(p_off.numpy(), p_act.numpy(), p_ts.numpy(), 12, nfa, flags=flags)
        ok, why = got.same_as(want)
        assert ok, (why, states, flags)


@pytest.mark.parametrize("flags", [0, abi.F_RETURN_ALL, abi.F_EVT_POS, abi.F_EVT_POS | abi.F_RETURN_ALL, abi.F_COUNT_MATCHES, abi.F_NO_EVENT_COLUMNS])
def test_patterns_without_kleene_states_on_traces_of_any_length(ctx, flags):
    """Kernel K1-L: 3-activity logs with 200 - 2 000 events per trace (every event is pattern-relevant, far beyond the 64 the
    mask kernels hold) against the oracle; the reference's engine has no per-trace limit (Engine.java:207-224)."""
    off, act, ts = gen.make_log(60, 200, 2000, 3, seed=9, max_gap_s=30, jitter_ms=True)
    short = gen.make_log(500, 0, 40, 3, seed=10, max_gap_s=30)           # the usual traces around them
    off = np.concatenate([off, off[-1] + short[0][1:]])
    act = np.concatenate([act, short[1]])
    ts = np.concatenate([ts, short[2]])
    patterns = [
        [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2])],
        [dict(kind=N_, types=[0]), dict(kind=X_, types=[1]), dict(kind=N_, types=[2], preds=[(abi.ATTR_POSITION, abi.OP_GE, 0, 4)])],
        [dict(kind=O_, types=[0, 1]), dict(kind=N_, types=[2], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 40)]),
         dict(kind=N_, types=[0], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 9), (abi.ATTR_TIMESTAMP, abi.OP_GE, 1, 5)])],
    ]
    for states in patterns:
        got = _check(ctx, off, act, ts, 3, states, flags)
        assert got.n_unsupported == 0 and got.n_traces > 0


NP1_SHAPES = [
    ("a b+ c", [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])]),
    ("a b+", [dict(kind=N_, types=[0]), dict(kind=P_, types=[1])]),
    ("a+ b", [dict(kind=P_, types=[0]), dict(kind=N_, types=[1])]),
    ("a (b|c) d+ (a|e) b", [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2]), dict(kind=P_, types=[3]), dict(kind=O_, types=[0, 4]), dict(kind=N_, types=[1])]),
    ("b b+ b", [dict(kind=N_, types=[1]), dict(kind=P_, types=[1]), dict(kind=N_, types=[1])]),
    ("a b+ c, gap within 6 (0,2)", [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]),
                                    dict(kind=N_, types=[2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 6)])]),
    ("a c b+ a, b within 200 s of a, last a at least 3 after c", [dict(kind=N_, types=[0]), dict(kind=N_, types=[2]),
        dict(kind=P_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 200)]), dict(kind=N_, types=[0], preds=[(abi.ATTR_POSITION, abi.OP_GE, 1, 3)])]),
    ("a b+ c, constraints dropped by onlyAppearances", [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]),
                                                         dict(kind=N_, types=[2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 3)])]),
]


@pytest.mark.parametrize("name,states", NP1_SHAPES, ids=[s[0] for s in NP1_SHAPES])
def test_one_kleene_plus_state_without_constraints_closed_form(ctx, name, states):
    """Class NP1 (detect_fast.cuh): the closed form replaces the run-list engine; occurrences, the engine's match count
    and the listed outliers (more than 64 relevant events) against the oracle, narrow and wide configuration."""
    only = abi.F_ONLY_APPEARANCES if "onlyAppearances" in name else 0
    for n_act, max_len in ((5, 30), (7, 120), (3, 90)):
        off, act, ts = gen.make_log(3000, 0, max_len, n_act, seed=77 + n_act, max_gap_s=100, jitter_ms=True)
        for flags in (0, abi.F_COUNT_MATCHES, abi.F_EVT_POS, abi.F_EVT_POS | abi.F_RETURN_ALL, abi.F_NO_EVENT_COLUMNS):
            got = _check(ctx, off, act, ts, n_act, states, flags | only)
            if n_act == 5:
                assert got.n_unsupported == 0
