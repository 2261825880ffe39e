"""The uniform placement (gather_uniform_kernel, csrc/detect.cu) against the CPU oracle, bit for bit.

When every matching trace holds one occurrence of k events, K1-P leaves two words per tile of 32 candidates (the lanes
that matched, the lanes it sent to the overflow list) and stages each reported event as one packed {pos, rank, act}
word plus its timestamp.  The placement takes the rows of K1-P's matches from those words and reads d_cnt / d_stage only
for the overflow lanes, which the staged kernels and K1-L answer.  The log here mixes both inside tiles: traces longer
than 64 slots, traces with more than 32 relevant events (both re-run on the staged kernels) and traces with more than
64 relevant events (K1-L) sit in the middle of tiles of K1-P traces; one tile matches on all 32 lanes and one holds only
overflow traces.  The trace count is not a multiple of 32 or 256 and exceeds 262 144, so the scan's second level runs.
The first traces are 64 events long and start on 8-event boundaries, so K1-P reports position 63, rank 63 (raw space)
and activity 254: the packed fields at their limits.

Every case asserts that it reaches the path it is about: K1-P runs (more launches than under SIESTA_K1_NO_NKP) and the
placement launched is gather_uniform_kernel (kernel names from torch.profiler)."""
import os

import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from tests import gen

pytestmark = pytest.mark.gpu

N_, X_, O_ = abi.STATE_NORMAL, abi.STATE_NEGATIVE, abi.STATE_OR
THREADS = max(1, min(32, os.cpu_count() or 1))
N_ACT = 255
N_TRACES = 300_011                  # not a multiple of 32 or 256, more than 262 144 candidates
EDGE_TRACES = 64                    # traces 0..63: 64 events each, the packed fields at their limits
FULL_TILE = 1000                    # candidates 32 000 .. 32 031 all match
OVF_TILE = 2000                     # candidates 64 000 .. 64 031 are all longer than 64 slots

GAP6 = [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
        dict(kind=X_, types=[3]), dict(kind=N_, types=[4]), dict(kind=N_, types=[5], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])]
# raw space (EventPos route with a position predicate): all 64 slots of an edge trace are relevant
EDGE = [dict(kind=N_, types=[253]), dict(kind=N_, types=[254], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 100)])]


def _chain(k):
    """k events over activities 0..6 (the eighth state repeats activity 0: K1-P takes at most seven signatures)."""
    return [dict(kind=N_, types=[i % 7]) for i in range(k)]


# (name, states, k, flags, candidate list?)
CASES = [
    ("k1", _chain(1), 1, 0, False),
    ("k2 evtpos", _chain(2), 2, abi.F_EVT_POS, False),
    ("k3 no columns", _chain(3), 3, abi.F_NO_EVENT_COLUMNS, False),
    ("gap6 k4", GAP6, 4, 0, False),
    ("gap6 k4 evtpos raw", GAP6, 4, abi.F_EVT_POS, False),
    ("gap6 k4 no columns", GAP6, 4, abi.F_NO_EVENT_COLUMNS, False),
    ("gap6 k4 candidates", GAP6, 4, 0, True),
    ("k5", _chain(5), 5, 0, False),
    ("k6 evtpos candidates", _chain(6), 6, abi.F_EVT_POS, True),
    ("k7 no columns", _chain(7), 7, abi.F_NO_EVENT_COLUMNS, False),
    ("k8", _chain(8), 8, 0, False),
    ("edge raw", EDGE, 2, abi.F_EVT_POS, False),
]


def _make_log(seed=0x0F1A7):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 41, size=N_TRACES).astype(np.int64)
    kind = np.zeros(N_TRACES, dtype=np.int8)        # 0 short, 1 > 64 slots, 2 > 32 relevant, 3 > 64 relevant, 4 edge, 5 full
    mid = np.arange(EDGE_TRACES + 5, N_TRACES, 97)   # every 97th trace: lands at every lane of a tile over the log
    kind[mid[0::3]] = 1
    kind[mid[1::3]] = 2
    kind[mid[2::3][::20]] = 3
    kind[:EDGE_TRACES] = 4
    kind[FULL_TILE * 32:FULL_TILE * 32 + 32] = 5
    kind[OVF_TILE * 32:OVF_TILE * 32 + 32] = 1
    lens[kind == 1] = rng.integers(70, 130, size=int((kind == 1).sum()))
    lens[kind == 2] = rng.integers(40, 60, size=int((kind == 2).sum()))
    lens[kind == 3] = rng.integers(500, 700, size=int((kind == 3).sum()))
    lens[kind == 4] = 64
    full_seq = np.array([0, 1, 4, 9, 5, 0, 1, 2, 3, 4, 5, 6, 0], dtype=np.int32)
    lens[kind == 5] = len(full_seq)
    off = np.zeros(N_TRACES + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    E = int(off[-1])
    trace_kind = np.repeat(kind, lens)
    act = rng.integers(0, 12, size=E).astype(np.int32)
    dense = (trace_kind == 2) | (trace_kind == 3)    # every event an activity of the patterns
    act[dense] = rng.integers(0, 7, size=int(dense.sum()))
    edge_ev = trace_kind == 4
    act[edge_ev] = 253
    act[off[1:EDGE_TRACES + 1] - 1] = 254           # the last slot (position 63) of every edge trace
    for t in np.flatnonzero(kind == 5):
        act[off[t]:off[t + 1]] = full_seq
    gaps = rng.integers(1, 301, size=E).astype(np.int64) * 1000
    ts = np.cumsum(gaps)
    first = np.repeat(off[:-1], lens)
    start = gen.T0_MS + rng.integers(0, 30 * 86400, size=N_TRACES).astype(np.int64) * 1000
    ts = ts - np.concatenate(([0], ts))[first] + np.repeat(start, lens)
    return off, act, ts.astype(np.int64), kind


def _launches():
    from sequencedetectionqueryexecutor_b200 import api
    return api.kernel_launches()


def _kernel_names(fn):
    """Names of the CUDA kernels fn launches, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _uses(names, kernel):
    return any(kernel in n for n in names)


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def mixed(ctx):
    off, act, ts, kind = _make_log()
    rng = np.random.default_rng(23)
    cand = np.sort(rng.choice(N_TRACES, size=N_TRACES // 2 + 7, replace=False)).astype(np.int64)
    assert len(cand) > 262_144 // 2 and len(cand) % 32
    wants = [oracle.detect(off, act, ts, abi.make_nfa(st), cand=cand if c else None, flags=fl, n_threads=THREADS)
             for _, st, _, fl, c in CASES]
    log = ctx.load_log(off, act, ts, N_ACT)
    yield off, act, ts, kind, cand, log, wants
    log.close()


def _tiles_of(want, n):
    hit = np.zeros(n, dtype=bool)
    hit[want.trace_idx] = True
    return hit


def test_mixed_tiles_equal_the_oracle(mixed, monkeypatch):
    off, act, ts, kind, cand, log, wants = mixed
    monkeypatch.delenv("SIESTA_NO_UNIFORM_GATHER", raising=False)
    monkeypatch.delenv("SIESTA_K1_NO_NKP", raising=False)
    mixed_tiles = 0
    for (name, st, k, fl, c), want in zip(CASES, wants):
        nfa = abi.make_nfa(st)
        cc = cand if c else None
        n0 = _launches()
        got, names = _kernel_names(lambda: log.detect(nfa, cand=cc, flags=fl))
        n_nkp = _launches() - n0
        ok, why = got.same_as(want)
        assert ok and got.n_unsupported == 0, (name, why)
        assert got.n_traces > 0 and got.n_events == got.n_traces * k, (name, got.n_traces, got.n_events)
        assert _uses(names, "gather_uniform_kernel"), (name, sorted(names))
        assert _uses(names, "detect_nkp_kernel") and _uses(names, "detect_long_kernel"), (name, sorted(names))
        monkeypatch.setenv("SIESTA_K1_NO_NKP", "1")
        n0 = _launches()
        log.detect(nfa, cand=cc, flags=fl)
        n_staged = _launches() - n0
        monkeypatch.delenv("SIESTA_K1_NO_NKP")
        assert n_nkp > n_staged, (name, "does not run on K1-P")
        if cc is None:
            hit = _tiles_of(want, N_TRACES)
            # tiles in which a K1-P match and a matching re-run trace (staged kernels or K1-L) sit side by side
            short = (kind == 0) & hit
            rerun = np.isin(kind, (1, 2, 3)) & hit
            pad = (-N_TRACES) % 32
            both = (np.concatenate([short, np.zeros(pad, bool)]).reshape(-1, 32).any(1) &
                    np.concatenate([rerun, np.zeros(pad, bool)]).reshape(-1, 32).any(1))
            mixed_tiles += int(both.sum())
            if name != "edge raw":
                assert hit[FULL_TILE * 32:FULL_TILE * 32 + 32].all(), (name, "the full tile does not match on every lane")
                assert hit[OVF_TILE * 32:OVF_TILE * 32 + 32].any(), (name, "no match in the overflow-only tile")
            if name == "gap6 k4":
                assert (hit & (kind == 3)).any(), "no K1-L trace matches"
    assert mixed_tiles > 1000, mixed_tiles


def test_packed_fields_at_their_limits(mixed):
    """Edge traces: K1-P reports position 63, rank 63 and activity 254, which take the packed word's fields to their
    largest values."""
    off, act, ts, kind, cand, log, wants = mixed
    i = [c[0] for c in CASES].index("edge raw")
    got = log.detect(abi.make_nfa(EDGE), flags=abi.F_EVT_POS)
    ok, why = got.same_as(wants[i])
    assert ok, why
    edge = got.trace_idx < EDGE_TRACES
    assert edge.sum() == EDGE_TRACES
    pos, rank, a = (np.asarray(getattr(got, c)).reshape(-1, 2)[edge] for c in ("ev_pos", "ev_rank", "ev_act"))
    assert (pos[:, 1] == 63).all() and (rank[:, 1] == 63).all() and (a[:, 1] == 254).all()


def test_uniform_request_without_k1p(mixed, monkeypatch):
    """SIESTA_K1_NO_NKP: every lane is an overflow lane, so the same placement reads d_cnt for every candidate."""
    off, act, ts, kind, cand, log, wants = mixed
    monkeypatch.setenv("SIESTA_K1_NO_NKP", "1")
    for (name, st, k, fl, c), want in zip(CASES, wants):
        if name not in ("gap6 k4", "gap6 k4 candidates", "k3 no columns", "k8"):
            continue
        got, names = _kernel_names(lambda: log.detect(abi.make_nfa(st), cand=cand if c else None, flags=fl))
        ok, why = got.same_as(want)
        assert ok and got.n_unsupported == 0, (name, why)
        assert _uses(names, "gather_uniform_kernel") and not _uses(names, "detect_nkp_kernel"), (name, sorted(names))


@pytest.mark.parametrize("flags", [0, abi.F_EVT_POS, abi.F_NO_EVENT_COLUMNS])
def test_compact_block_equals_the_resident_result(ctx, flags):
    """The exchange's compact block on one device (world 1), placed by gather_uniform_kernel<true>, decodes to the
    resident result of the same request."""
    from sequencedetectionqueryexecutor_b200 import api
    from sequencedetectionqueryexecutor_b200 import distributed as D
    off, act, ts, kind = _make_log(0xB10C5)
    n = 20_011
    e1 = int(off[n])
    off, act, ts = off[:n + 1], act[:e1], ts[:e1]
    nfa = abi.make_nfa(GAP6)
    log = ctx.load_log(off, act, ts, N_ACT)
    try:
        want = log.detect(nfa, flags=flags)
        ok, why = want.same_as(oracle.detect(off, act, ts, nfa, flags=flags, n_threads=THREADS))
        assert ok, why
        x = api.Exchange(ctx, 1, 0, api.exchange_required_bytes(log, nfa, flags))
        try:
            (dm, _), names = _kernel_names(lambda: x.detect_allgather(log, nfa, flags))
            try:
                got = D.to_match_result(dm.tensors(0), dm.n_matches_emitted)
            finally:
                dm.close()
        finally:
            x.close()
        assert _uses(names, "gather_uniform_kernel") and _uses(names, "detect_nkp_kernel"), sorted(names)
        ok, why = got.same_as(want)
        assert ok and want.n_traces > 0, why
    finally:
        log.close()
