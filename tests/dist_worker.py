"""Worker of tests/test_distributed_cpu.py: launched by torch.distributed.run with the gloo backend on CPU.
Each rank computes the counts of its shard with the ORACLE (test infrastructure standing in for the GPU kernels, which
need a device), then combines them with the product's all-reduce code; rank 0 compares with the unsharded oracle
result."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from sequencedetectionqueryexecutor_b200 import distributed as D  # noqa: E402
from tests import gen  # noqa: E402


def main():
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    off, act, ts = gen.make_log(1500, 0, 40, 8, seed=2024)
    l_off, l_act = D.local_shard(off, act, ts, rank, world)[:2]
    lc = oracle.declare_counts(l_off, l_act, 8, 40)
    packed = D.allreduce_counts(torch.from_numpy(lc.packed.copy()))
    wc = oracle.declare_counts(off, act, 8, 40)
    ok_declare = bool(np.array_equal(packed.numpy(), wc.packed))
    # pair statistics: per-shard records (oracle) packed like siesta_pair_stats_device, combined by the product code
    pairs = [(0, 1), (1, 0), (2, 2), (7, 3)]

    def pack(recs):
        rows = []
        for r in recs:
            sq = r["sum_squares"]
            rows.append([r["count"], r["sum"], r["min"] if r["count"] else 2 ** 63 - 1, r["max"] if r["count"] else -2 ** 63,
                         sq & 0xFFFFFFFF, (sq >> 32) & 0xFFFFFFFF, (sq >> 64) & 0xFFFFFFFF, (sq >> 96) & 0xFFFFFFFF])
        return torch.tensor(rows, dtype=torch.int64).reshape(-1)

    # long gaps so that the squares need the upper limbs
    big_ts = ts * 1000
    l_big = big_ts[int(off[D.shard_bounds(off, world)[rank]]):int(off[D.shard_bounds(off, world)[rank + 1]])]
    st = D.allreduce_pair_stats(pack(oracle.pair_stats(l_off, l_act, l_big, pairs)))
    ok_stats = D.pair_stats_records(st) == oracle.pair_stats(off, act, big_ts, pairs)
    b = D.shard_bounds(off, world)
    ev = [int(off[b[r + 1]] - off[b[r]]) for r in range(world)]
    if rank == 0:
        with open(sys.argv[1], "w") as f:
            json.dump({"ok_declare": ok_declare, "ok_stats": bool(ok_stats), "world": world,
                       "bounds": [int(x) for x in b], "events_per_rank": ev}, f)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
