"""A pair index that follows a growing log (siesta_index_refresh / siesta_index_append, csrc/intersect.cu): one JSON line.

Size: the flagship's 100 M traces x 50 events (bench.make_log_device, generated on the GPU; --traces 10000000 for the
10 M size), the 9 distinct true pairs of configs[4] (two OR-expansions of 6 pairs each, three of them shared), and the
batch of tools/bench_log_append.py: 1 M touched traces x 5 events plus 1 M new traces x 50 events.  Timed, each the
median of --repeats calls after one warm-up:
  refresh   siesta_index_refresh of the built index onto the appended log (call time, host clock; and kernel_ms)
  build     siesta_index_build on the appended log (call time), what a caller without refresh runs
  append    siesta_index_append of the batch's delta lists from host memory onto an index of the old lists (kernel_ms and
            call time)
  reload    siesta_index_load of the full union lists from pinned host memory (call time), what append replaces
  copy_     a torch copy_ of the new lists' bytes in the same run: the in-run ceiling of the merge
Algorithmic bytes: merge = 8 B x (sum |old| + sum |new| + sum |delta|); refresh adds 4 B per event of the listed traces,
16 B per listed trace and 2 x n_pairs flag bytes per listed trace.  Parity: refreshed lists == rebuilt lists, appended
lists == the union of the old and delta lists (np.union1d up to 10 M traces, the same union by sorted insertion above),
every list compared in full.  Comparison indexes are freed as soon as they are checked: the two logs take about 123 GB.
`python tools/bench_index_append.py [--traces N] [--touched N] [--new N] [--repeats N]`"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_log_append import GAP_S, LENGTH, N_ACT, SEED, card, make_batch  # noqa: E402
from sequencedetectionqueryexecutor_b200 import api  # noqa: E402
from sequencedetectionqueryexecutor_b200._lib import check, lib  # noqa: E402

# configs[4]: A (B | C) !D E F -> expansions A B E F and A C E F, each with the 6 ordered pairs of its 4 events
PAIRS = [(0, 1), (0, 4), (0, 5), (1, 4), (1, 5), (4, 5), (0, 2), (2, 4), (2, 5)]


def median_call(fn, repeats, keep_last=True):
    """fn() -> (obj, kernel_ms or None) with obj closed between calls; first call is the warm-up.
    -> (last obj, [call ms], [kernel ms])"""
    obj, calls, kern = None, [], []
    for r in range(repeats + 1):
        if obj is not None:
            obj.close()
        t0 = time.perf_counter()
        obj, ms = fn()
        dt = (time.perf_counter() - t0) * 1e3
        if r:
            calls.append(dt)
            if ms is not None:
                kern.append(ms)
    if not keep_last:
        obj.close()
        obj = None
    return obj, calls, kern


def sorted_union(a, b):
    """Union of two ascending duplicate-free arrays by sorted insertion (linear; np.union1d sorts)."""
    pos = np.searchsorted(a, b)
    held = np.zeros(len(b), dtype=bool)
    inside = pos < len(a)
    held[inside] = a[pos[inside]] == b[inside]
    return np.insert(a, pos[~held], b[~held])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--traces", type=int, default=100_000_000)
    ap.add_argument("--touched", type=int, default=None, help="default: 1 %% of --traces")
    ap.add_argument("--new", type=int, default=None, help="default: 1 %% of --traces")
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_index_append: no CUDA device")
    T = args.traces
    touched = args.touched if args.touched is not None else max(T // 100, 1)
    n_new = args.new if args.new is not None else max(T // 100, 1)
    name, power = card()
    dev = torch.device("cuda", 0)
    ctx = api.Context(0)
    d_off, d_act, d_ts = bench.make_log_device(torch, dev, 0, T, T, LENGTH, N_ACT, SEED, GAP_S)
    base = ctx.wrap_log(d_off, d_act, d_ts, N_ACT, max_trace_len=LENGTH)
    idx, boff, bact, bts = make_batch(torch, d_ts, T, touched, 5, n_new, 50, seed=T)
    new_log, _ = base.append(idx, boff, bact, bts, n_new_traces=n_new)
    torch.cuda.synchronize()
    old = base.build_index(PAIRS)
    n_pairs = len(PAIRS)
    old_len = [int(lib().siesta_index_list_len(old._h, p)) for p in range(n_pairs)]

    # refresh vs build on the new log
    refreshed, refresh_call, refresh_kern = median_call(lambda: old.refresh(new_log, idx), args.repeats)
    rebuilt, build_call, _ = median_call(lambda: (new_log.build_index(PAIRS), None), args.repeats)
    new_lists = [refreshed.posting_list(p) for p in range(n_pairs)]
    refresh_ok = all(np.array_equal(new_lists[p], rebuilt.posting_list(p)) for p in range(n_pairs))
    rebuilt.close()
    refreshed.close()
    new_len = [len(x) for x in new_lists]

    # the batch's delta lists (what its index.parquet rows hold): the new lists restricted to the listed traces
    delta = []
    for x in new_lists:
        pos = np.minimum(np.searchsorted(x, idx), max(len(x) - 1, 0))
        delta.append(idx[x[pos] == idx] if len(x) else np.zeros(0, np.int64))
    del new_lists
    delta_len = [len(x) for x in delta]
    appended, append_call, append_kern = median_call(lambda: old.append(new_log, delta), args.repeats)
    union_ok = True
    for p in range(n_pairs):
        o = old.posting_list(p)
        want = np.union1d(o, delta[p]) if T <= 10_000_000 else sorted_union(o, delta[p])
        union_ok &= bool(np.array_equal(appended.posting_list(p), want))
    del o, want

    # reload: siesta_index_load of the full union lists from pinned host memory
    n_total = sum(new_len)
    h_flat = torch.empty(max(n_total, 1), dtype=torch.int64, pin_memory=True).numpy()
    h_off = np.zeros(n_pairs + 1, dtype=np.int64)
    np.cumsum(new_len, out=h_off[1:])
    for p in range(n_pairs):
        check(lib().siesta_index_get_list(appended._h, p, api._ptr(h_flat[h_off[p]:]), new_len[p]))
    appended.close()
    pa = np.array([a for a, _ in PAIRS], dtype=np.int32)
    pb = np.array([b for _, b in PAIRS], dtype=np.int32)

    def reload():
        h = C.c_void_p()
        check(lib().siesta_index_load(new_log._h, n_pairs, api._ptr(pa), api._ptr(pb), api._ptr(h_off), api._ptr(h_flat), C.byref(h)))
        return old._adopt(new_log, h), None

    _, reload_call, _ = median_call(reload, args.repeats, keep_last=False)
    del h_flat
    old.close()

    # in-run ceiling: copy_ of the new lists' bytes
    src = torch.empty(n_total, dtype=torch.int64, device=dev)
    dst = torch.empty_like(src)
    cp = []
    for r in range(args.repeats + 1):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        dst.copy_(src)
        s1.record()
        torch.cuda.synchronize()
        if r:
            cp.append(s0.elapsed_time(s1))
    del src, dst
    torch.cuda.empty_cache()
    new_log.close()
    base.close()
    ctx.close()

    k = len(idx)
    listed_events = int(boff[-1]) + LENGTH * int(np.count_nonzero(idx < T))
    merge_bytes = 8 * (sum(old_len) + sum(new_len) + sum(delta_len))
    refresh_bytes = merge_bytes + 4 * listed_events + 16 * k + 2 * n_pairs * k
    med = lambda v: float(np.median(v))   # noqa: E731
    copy_ms = med(cp)
    out = {"kernels": "pair_flags_kernel (work list) + compaction + index_dup_kernel + index_merge_kernel",
           "traces": T, "events": T * LENGTH, "pairs": n_pairs, "listed_traces": k, "touched_traces": touched, "new_traces": n_new,
           "batch_events": int(boff[-1]), "old_list_entries": sum(old_len), "new_list_entries": sum(new_len),
           "delta_entries": sum(delta_len),
           "refresh_call_ms": med(refresh_call), "refresh_kernel_ms": med(refresh_kern), "refresh_call_ms_all": refresh_call,
           "build_call_ms": med(build_call), "build_call_ms_all": build_call,
           "refresh_over_build": med(refresh_call) / med(build_call),
           "append_kernel_ms": med(append_kern), "append_call_ms": med(append_call), "append_kernel_ms_all": append_kern,
           "reload_call_ms": med(reload_call), "reload_call_ms_all": reload_call,
           "reload_over_append_call": med(reload_call) / med(append_call),
           "copy_ms": copy_ms, "copy_bytes": 16 * sum(new_len), "append_kernel_over_copy": med(append_kern) / copy_ms,
           "merge_algorithmic_bytes": merge_bytes, "append_algorithmic_GBps": merge_bytes / (med(append_kern) * 1e-3) / 1e9,
           "refresh_algorithmic_bytes": refresh_bytes, "refresh_algorithmic_GBps": refresh_bytes / (med(refresh_kern) * 1e-3) / 1e9,
           "copy_GBps": 16 * sum(new_len) / (copy_ms * 1e-3) / 1e9,
           "parity_refresh_equals_build": bool(refresh_ok), "parity_append_equals_union": bool(union_ok),
           "gpu": name, "power_limit": power}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
