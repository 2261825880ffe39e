"""Launch schedules and alternate kernels of /detection that the small logs of the other suites never reach, each
compared with the CPU oracle bit for bit.

Kernel K1-P (detect_nkp.cu) hands tiles of 32 traces to its warps `tile_batch` at a time (1, 2 or 4, picked from the
tiles per warp) and passes the next batch from warp to warp through `next_batch` / `next_batch2`.  A log of a few
thousand traces always runs with batch 1 and one tile per warp, so here the batch and the grid are forced through the
launchers' tuning knobs on a log of about 300 000 traces, and the production choice (batch 4, picked by the launcher)
is reached at about 1.3 M traces with one CTA per SM.  The knobs that switch kernels (SIESTA_K1_NO_NKP,
SIESTA_K1_NO_LONG) or shrink the staged kernel's CTA (SIESTA_K1_THREADS) are covered at small size.

Every case asserts from the device's SM count and the launchers' constants that it reaches the schedule it is about,
so a change to a constant fails here instead of quietly shrinking the coverage."""
import os

import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200._lib import SiestaError
from tests import gen

pytestmark = pytest.mark.gpu

N_, P_, S_, X_, O_ = abi.STATE_NORMAL, abi.STATE_KLEENE_PLUS, abi.STATE_KLEENE_STAR, abi.STATE_NEGATIVE, abi.STATE_OR
NT = 128              # threads per CTA of K1 / K1-P (detect_common.cuh)
THREADS = max(1, min(32, os.cpu_count() or 1))   # oracle threads


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _oracle(off, act, ts, states, flags, cand=None):
    return oracle.detect(off, act, ts, abi.make_nfa(states), cand=cand, flags=flags, n_threads=THREADS)


def _launches():
    from sequencedetectionqueryexecutor_b200 import api
    return api.kernel_launches()


@pytest.fixture(scope="module")
def ctx():
    from sequencedetectionqueryexecutor_b200 import api
    c = api.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ K1-P tile scheduler
# class NK patterns with 1, 2-3 and 4-7 activity signatures (one, two and three bit planes); Markov ones (every predicate
# reads the previous positive state) and non-Markov ones; a negative state
ONE_SIG = [dict(kind=N_, types=[0]), dict(kind=N_, types=[0], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 5)])]
THREE_SIG = [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 6)]),
             dict(kind=N_, types=[3])]
FIVE_SIG_NEG = [dict(kind=N_, types=[0]), dict(kind=O_, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
                dict(kind=X_, types=[3]), dict(kind=N_, types=[4]),
                dict(kind=N_, types=[5], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])]
FOUR_SIG_NON_MARKOV = [dict(kind=N_, types=[0]), dict(kind=N_, types=[1]), dict(kind=N_, types=[2]),
                       dict(kind=N_, types=[3], preds=[(abi.ATTR_POSITION, abi.OP_GE, 0, 4)])]
SEVEN_SIG_NON_MARKOV = [dict(kind=N_, types=[k], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 14)] if k == 3 else [])
                        for k in range(7)]


def _no_preds(states):
    return [dict(kind=s["kind"], types=s["types"]) for s in states]


# (name, states, flags, candidate list?) - rank space: EventTs route with position predicates, or EventPos without any;
# raw space: EventPos with position predicates
NKP_CASES = [
    ("rank 1 plane", ONE_SIG, 0, False),
    ("rank 2 planes markov", THREE_SIG, 0, False),
    ("rank 3 planes markov negative", FIVE_SIG_NEG, 0, False),
    ("rank 3 planes non-markov count", FOUR_SIG_NON_MARKOV, abi.F_COUNT_MATCHES, False),
    ("rank 3 planes non-markov returnAll", SEVEN_SIG_NON_MARKOV, abi.F_RETURN_ALL, False),
    ("rank evtpos no predicates", _no_preds(FIVE_SIG_NEG), abi.F_EVT_POS, False),
    ("raw 3 planes markov negative", FIVE_SIG_NEG, abi.F_EVT_POS, False),
    ("raw 3 planes non-markov no columns", FOUR_SIG_NON_MARKOV, abi.F_EVT_POS | abi.F_NO_EVENT_COLUMNS, False),
    ("raw 1 plane count", ONE_SIG, abi.F_EVT_POS | abi.F_COUNT_MATCHES, False),
    ("raw 2 planes returnAll candidates", THREE_SIG, abi.F_EVT_POS | abi.F_RETURN_ALL, True),
    ("rank 3 planes candidates", SEVEN_SIG_NON_MARKOV, 0, True),
]


@pytest.fixture(scope="module")
def nkp_log(ctx):
    """About 300 000 traces of 0 - 80 events (some beyond K1-P's 64 slots or 32 relevant events: they move to the staged
    kernel in the same request).  The trace count is not a multiple of 32, and the event count not a multiple of 8, so
    the end sector of the last trace lies past the log's end.  Oracle results are computed once per case."""
    for seed in range(0x5C4ED, 0x5C4ED + 64):
        off, act, ts = gen.make_log(300_007, 0, 80, 12, seed=seed, max_gap_s=300)
        if len(act) % 8 and off[-1] > off[-2]:
            break
    assert (len(off) - 1) % 32 and len(act) % 8 and off[-1] > off[-2]
    rng = np.random.default_rng(17)
    cand = np.sort(rng.choice(len(off) - 1, size=(len(off) - 1) // 2, replace=False)).astype(np.int64)
    log = ctx.load_log(off, act, ts, 12)
    wants = [_oracle(off, act, ts, st, fl, cand if c else None) for _, st, fl, c in NKP_CASES]
    yield off, act, ts, cand, log, wants
    log.close()


def _detect_counting(log, states, flags, cand):
    n0 = _launches()
    got = log.detect(abi.make_nfa(states), cand=cand, flags=flags)
    return got, _launches() - n0


def test_nkp_runs_for_every_case_and_equals_the_staged_kernel(nkp_log, monkeypatch):
    """Every case of the matrix below runs on K1-P: without SIESTA_K1_NO_NKP a request launches more kernels.  With
    the knob every trace runs on the staged kernel, and both equal the oracle."""
    off, act, ts, cand, log, wants = nkp_log
    for (name, st, fl, c), want in zip(NKP_CASES, wants):
        cc = cand if c else None
        got, n_nkp = _detect_counting(log, st, fl, cc)
        ok, why = got.same_as(want)
        assert ok and got.n_unsupported == 0, (name, why)
        monkeypatch.setenv("SIESTA_K1_NO_NKP", "1")
        got2, n_staged = _detect_counting(log, st, fl, cc)
        monkeypatch.delenv("SIESTA_K1_NO_NKP")
        ok, why = got2.same_as(want)
        assert ok, (name, "SIESTA_K1_NO_NKP", why)
        assert n_nkp > n_staged, (name, n_nkp, n_staged)


@pytest.mark.parametrize("batch", [1, 2, 3, 4])
@pytest.mark.parametrize("ctas_per_sm", [None, 1])
@pytest.mark.parametrize("evaluator", ["default", "no-markov"])
def test_nkp_tile_batches_grids_and_evaluators_equal_the_oracle(nkp_log, monkeypatch, batch, ctas_per_sm, evaluator):
    """SIESTA_NKP_TILE_BATCH x SIESTA_K1_CTAS_PER_SM x evaluator.  With one CTA per SM every warp takes at least three
    batches of the log-wide cases, so the hand-off of both next_batch and next_batch2 runs; with the default grid the
    tiles run out while most warps still hold their first batch (the tail of the schedule)."""
    off, act, ts, cand, log, wants = nkp_log
    n_tiles = (len(off) - 1 + 31) // 32
    if ctas_per_sm == 1:
        warps = _sms() * ctas_per_sm * (NT // 32)
        assert n_tiles // warps >= 3 * batch, "the log no longer gives every warp three batches"
        monkeypatch.setenv("SIESTA_K1_CTAS_PER_SM", str(ctas_per_sm))
    else:
        monkeypatch.delenv("SIESTA_K1_CTAS_PER_SM", raising=False)
    monkeypatch.setenv("SIESTA_NKP_TILE_BATCH", str(batch))
    if evaluator == "no-markov":
        monkeypatch.setenv("SIESTA_NKP_NO_MARKOV", "1")
    else:
        monkeypatch.delenv("SIESTA_NKP_NO_MARKOV", raising=False)
    for (name, st, fl, c), want in zip(NKP_CASES, wants):
        got = log.detect(abi.make_nfa(st), cand=cand if c else None, flags=fl)
        ok, why = got.same_as(want)
        assert ok and got.n_unsupported == 0, (name, why)


def test_nkp_production_schedule_picks_batch_four(ctx, monkeypatch):
    """No batch override, one CTA per SM, about 1.3 M traces of 0 - 12 events: launch_one picks tile_batch 4 by itself
    (per_warp = n_tiles / (grid * NT / 32) >= 64), the schedule of the 100 M-trace benchmark."""
    sms = _sms()
    warps = sms * 1 * (NT // 32)
    n = warps * 32 * 70 + 13                 # 70 tiles per warp: batch 4 with margin, and not a multiple of 32
    off, act, ts = gen.make_log(n, 0, 12, 8, seed=0x13A7C4, max_gap_s=300)
    n_tiles = (n + 31) // 32
    grid = min((n_tiles + NT // 32 - 1) // (NT // 32), sms * 1)
    per_warp = n_tiles // (grid * (NT // 32))
    assert per_warp >= 64, per_warp           # launch_one: per_warp >= 64 -> tile_batch 4
    monkeypatch.setenv("SIESTA_K1_CTAS_PER_SM", "1")
    monkeypatch.delenv("SIESTA_NKP_TILE_BATCH", raising=False)
    rng = np.random.default_rng(5)
    cand = np.sort(rng.choice(n, size=n * 19 // 20, replace=False)).astype(np.int64)   # 95 %: still batch 4
    assert ((len(cand) + 31) // 32) // (grid * (NT // 32)) >= 64
    log = ctx.load_log(off, act, ts, 8)
    try:
        for st, fl, c in ((FIVE_SIG_NEG, 0, None), (THREE_SIG, abi.F_EVT_POS, None), (FOUR_SIG_NON_MARKOV, abi.F_COUNT_MATCHES, None),
                          (ONE_SIG, abi.F_EVT_POS | abi.F_RETURN_ALL, cand)):
            got, n_nkp = _detect_counting(log, st, fl, c)
            ok, why = got.same_as(_oracle(off, act, ts, st, fl, c))
            assert ok, (st, fl, why)
            monkeypatch.setenv("SIESTA_K1_NO_NKP", "1")
            _, n_staged = _detect_counting(log, st, fl, c)
            monkeypatch.delenv("SIESTA_K1_NO_NKP")
            assert n_nkp > n_staged, "the case does not run on K1-P"
    finally:
        log.close()


# ------------------------------------------------------------------------------------------------ the remaining knobs
def _check(ctx, off, act, ts, n_act, states, flags, cand=None):
    """Device result against the oracle: traces listed as unsupported are left out, every other trace is exact."""
    nfa = abi.make_nfa(states)
    log = ctx.load_log(off, act, ts, n_act)
    try:
        n0 = _launches()
        got = log.detect(nfa, cand=cand, flags=flags)
        n_launch = _launches() - n0
    finally:
        log.close()
    want = oracle.detect(off, act, ts, nfa, cand=cand, flags=flags)
    if got.n_unsupported:
        out = set(got.unsupported_trace_idx.tolist())
        assert got.as_dict() == {t: o for t, o in want.as_dict().items() if t not in out}, (states, flags)
        assert got.err_trace_idx.tolist() == [t for t in want.err_trace_idx.tolist() if t not in out]
    else:
        ok, why = got.same_as(want)
        assert ok, (why, states, flags)
    return got, n_launch


CONFIG5 = FIVE_SIG_NEG


def _knob_cases(seed):
    """test_raw_slot_kernel_nk_class-style requests: random NK NFAs over traces on both sides of the 64-slot limit, then
    the config-5 shape on traces of 0 - 130 events."""
    from tests import soak_fast
    rng = np.random.default_rng(seed)
    out = []
    for it in range(24):
        n_act = int(rng.choice([3, 5, 8, 20, 40, 64]))
        lo, hi = [(0, 30), (40, 70), (55, 66), (0, 130)][it % 4]
        log = gen.make_log(700, lo, hi, n_act, seed=int(rng.integers(1 << 30)), max_gap_s=300)
        states = soak_fast.nk_nfa(rng, min(n_act, 8))
        for st in states:   # time predicates only on the EventPos route (elsewhere they need relative seconds)
            st["preds"] = [p for p in st["preds"] if p[0] == abi.ATTR_POSITION or it % 2 == 0]
        flags = abi.F_EVT_POS if it % 2 == 0 else 0
        if rng.random() < 0.3:
            flags |= abi.F_COUNT_MATCHES
        if rng.random() < 0.2:
            flags |= abi.F_NO_EVENT_COLUMNS
        cand = np.sort(rng.choice(700, size=300, replace=False)).astype(np.int64) if rng.random() < 0.3 else None
        out.append((log, n_act, states, flags, cand))
    c5 = gen.make_log(3000, 0, 130, 20, seed=seed + 1)
    for flags in (0, abi.F_RETURN_ALL, abi.F_EVT_POS, abi.F_EVT_POS | abi.F_RETURN_ALL):
        out.append((c5, 20, CONFIG5, flags, None))
    return out


@pytest.mark.parametrize("knob", ["SIESTA_K1_NO_NKP", "SIESTA_K1_NO_LONG"])
def test_kernel_switch_knobs_equal_the_oracle(ctx, monkeypatch, knob):
    """SIESTA_K1_NO_NKP sends class NK to the staged kernel; SIESTA_K1_NO_LONG drops kernel K1-L, so traces beyond the
    mask kernels' limits are listed as unsupported instead.  Each request with the knob launches a different number of
    kernels than without it (the knob is read), and every result equals the oracle."""
    monkeypatch.delenv(knob, raising=False)
    switched = 0
    n_unsup = 0
    for log, n_act, states, flags, cand in _knob_cases(9300):
        try:
            _, n_plain = _check(ctx, *log, n_act, states, flags, cand)
        except SiestaError as e:
            assert e.code == abi.E_UNSUPPORTED
            continue
        monkeypatch.setenv(knob, "1")
        try:
            got, n_knob = _check(ctx, *log, n_act, states, flags, cand)
        except SiestaError as e:
            assert e.code == abi.E_UNSUPPORTED
            continue
        finally:
            monkeypatch.delenv(knob)
        switched += n_knob != n_plain
        n_unsup += got.n_unsupported
    assert switched >= 8, switched
    if knob == "SIESTA_K1_NO_LONG":
        assert n_unsup > 0, "no trace went beyond the mask kernels: K1-L was never needed"


@pytest.mark.parametrize("threads", [32, 64])
def test_staged_kernel_with_fewer_threads_per_cta(ctx, monkeypatch, threads):
    """SIESTA_K1_THREADS: the staged kernel with one or two warps per CTA.  Under SIESTA_K1_NO_NKP every class NK trace
    runs on it, so its grid covers the whole request."""
    monkeypatch.setenv("SIESTA_K1_NO_NKP", "1")
    monkeypatch.setenv("SIESTA_K1_THREADS", str(threads))
    assert threads % 32 == 0 and threads < NT
    n_ok = 0
    for log, n_act, states, flags, cand in _knob_cases(9400 + threads):
        try:
            _check(ctx, *log, n_act, states, flags, cand)
        except SiestaError as e:
            assert e.code == abi.E_UNSUPPORTED
            continue
        n_ok += 1
    assert n_ok >= 14
    # a Kleene shape (run-list engine) and the NP1 closed form as well
    off, act, ts = gen.make_log(4000, 0, 90, 6, seed=9500 + threads, max_gap_s=120, jitter_ms=True)
    _check(ctx, off, act, ts, 6, [dict(kind=P_, types=[0]), dict(kind=S_, types=[1], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], 0)
    _check(ctx, off, act, ts, 6, [dict(kind=N_, types=[0]), dict(kind=P_, types=[1]), dict(kind=N_, types=[2])], abi.F_RETURN_ALL)
