"""The multi-GPU host plumbing on CPU: shard bounds, per-shard results joined in rank order, and world_size-2 (and 3)
gloo runs of the count all-reduces."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from sequencedetectionqueryexecutor_b200 import _abi as abi
from sequencedetectionqueryexecutor_b200 import distributed as D
from tests import gen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_bounds_cover_and_balance():
    rng = np.random.default_rng(0)
    lens = rng.integers(0, 60, size=1000)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    for world in (1, 2, 3, 8):
        b = D.shard_bounds(off, world)
        assert b[0] == 0 and b[-1] == 1000 and np.all(np.diff(b) >= 0) and len(b) == world + 1
        ev = np.array([off[b[r + 1]] - off[b[r]] for r in range(world)])
        assert ev.sum() == off[-1] and ev.max() - ev.min() <= 2 * 60
    assert D.shard_bounds(np.zeros(1, dtype=np.int64), 4).tolist() == [0, 0, 0, 0, 0]


def test_local_shards_joined_in_rank_order_equal_the_whole_log():
    """Every rank's shard detected on its own, with trace indices shifted by the shard's first trace and the columns
    concatenated in rank order, is the match list of the whole log."""
    off, act, ts = gen.make_log(1500, 0, 40, 8, seed=2024)
    nfa = abi.make_nfa([dict(kind=abi.STATE_NORMAL, types=[0]), dict(kind=abi.STATE_KLEENE_PLUS, types=[1]),
                        dict(kind=abi.STATE_NORMAL, types=[2], preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 3000)])])
    want = oracle.detect(off, act, ts, nfa, flags=abi.F_RETURN_ALL)
    assert want.n_traces > 10
    for world in (1, 2, 3, 8):
        parts = []
        for rank in range(world):
            l_off, l_act, l_ts, first = D.local_shard(off, act, ts, rank, world)
            parts.append((oracle.detect(l_off, l_act, l_ts, nfa, flags=abi.F_RETURN_ALL), first))
        got = {k: np.concatenate([getattr(p, k) + first for p, first in parts]) for k in ("trace_idx", "err_trace_idx")}
        for k in ("occ_off", "ev_off"):
            got[k] = np.concatenate(([0], np.cumsum(np.concatenate([np.diff(getattr(p, k)) for p, _ in parts]))))
        for k in ("ev_pos", "ev_rank", "ev_act", "ev_ts_ms"):
            got[k] = np.concatenate([getattr(p, k) for p, _ in parts])
        for k, v in got.items():
            assert np.array_equal(v, getattr(want, k)), (world, k)


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_allreduce_counts_and_pair_stats(world, tmp_path):
    out = tmp_path / "r.json"
    port = 29650 + world
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py"), str(out)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads(out.read_text())
    assert res["world"] == world
    assert res["ok_declare"] and res["ok_stats"]
