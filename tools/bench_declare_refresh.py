"""The /declare counts that follow a growing log (siesta_declare_counts_refresh, csrc/declare.cu): one JSON line per alphabet.

Size: the flagship's fixed-length synthetic log, 100 M traces x 50 events (bench.make_log_device, generated on the GPU;
--traces 10000000 for the 10 M size), and the batch of tools/bench_log_append.py: 1 % touched traces x 5 events plus 1 %
new traces x 50 events (--dense-traces: every trace touched, 1 % new).  The log is generated once over 400 activities;
the alphabets 400, 100 and 20 follow in place by `act %= A` (400 and 100 are multiples of the next alphabet, so each
stays uniform).  Timed per alphabet, each the median of --repeats calls after one warm-up:
  refresh   siesta_declare_counts_refresh(old log -> appended log) from the old counts (kernel_ms; call time, host clock)
  full      siesta_declare_counts on the appended log (kernel_ms; call time): what a caller without the refresh runs
  ceiling   siesta_declare_counts on a log built from only the listed traces' old and new versions (kernel_ms) plus a
            torch copy_ of the result's bytes: the in-run ceiling of the refresh (its counting work, one pass over the array)
Algorithmic bytes of the refresh: 4 B per event of the listed traces in both logs, 8 B per listed trace, the count array
read twice (old, delta) and written once, 16 B per old trace for the length check.  Parity: refresh == full, every value.
`python tools/bench_declare_refresh.py [--traces N] [--dense-traces] [--alphabets 400,100,20] [--repeats N] [--out FILE]`"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_log_append import GAP_S, LENGTH, SEED, card  # noqa: E402
from sequencedetectionqueryexecutor_b200 import api  # noqa: E402

K_CAP = 64
A_GEN = 400


def make_batch(torch, d_ts, T, touched_idx, touched_len, new, new_len, seed):
    """Touched traces (ascending) get `touched_len` events after their last one, new traces `new_len`; ids over A_GEN."""
    rng = np.random.default_rng(seed)
    tt = np.asarray(touched_idx, dtype=np.int64)
    last = d_ts[torch.from_numpy(tt * LENGTH + LENGTH - 1).to(d_ts.device)].cpu().numpy()
    idx = np.concatenate((tt, T + np.arange(new, dtype=np.int64)))
    lens = np.concatenate((np.full(len(tt), touched_len), np.full(new, new_len))).astype(np.int64)
    off = np.zeros(len(idx) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    act = rng.integers(0, A_GEN, size=int(off[-1]), dtype=np.int32)
    gaps = rng.integers(1, GAP_S + 1, size=int(off[-1]), dtype=np.int64) * 1000
    start = np.concatenate((last, 1577836800000 + rng.integers(0, 30 * 86400, size=new, dtype=np.int64) * 1000))
    seg_start = np.repeat(off[:-1], lens)
    cs = np.cumsum(gaps)
    ts = cs - np.concatenate(([0], cs))[seg_start] + np.repeat(start, lens)
    return idx, off, act, ts


def timed(fn, repeats):
    """fn() -> (result, kernel_ms); first call is the warm-up -> (last result, [call ms], [kernel ms])"""
    res, calls, kern = None, [], []
    for r in range(repeats + 1):
        t0 = time.perf_counter()
        res, ms = fn()
        dt = (time.perf_counter() - t0) * 1e3
        if r:
            calls.append(dt)
            kern.append(ms)
    return res, calls, kern


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--traces", type=int, default=100_000_000)
    ap.add_argument("--dense-traces", action="store_true", help="touch every trace (5 events each) instead of 1 %%")
    ap.add_argument("--alphabets", default="400,100,20")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_declare_refresh: no CUDA device")
    alphabets = [int(a) for a in args.alphabets.split(",")]
    assert all(A_GEN % a == 0 for a in alphabets) and all(alphabets[i] % alphabets[i + 1] == 0 for i in range(len(alphabets) - 1))
    T = args.traces
    n_new = max(T // 100, 1)
    rng = np.random.default_rng(T)
    touched_idx = np.arange(T, dtype=np.int64) if args.dense_traces else np.sort(rng.choice(T, size=max(T // 100, 1), replace=False))
    name, power = card()
    dev = torch.device("cuda", 0)
    ctx = api.Context(0)
    d_off, d_act, d_ts = bench.make_log_device(torch, dev, 0, T, T, LENGTH, A_GEN, SEED, GAP_S)
    idx, boff, bact, bts = make_batch(torch, d_ts, T, touched_idx, 5, n_new, 50, seed=T + 1)
    k, k_t = len(idx), len(touched_idx)
    d_tt = torch.from_numpy(touched_idx).to(dev)
    lines = []
    for A in alphabets:
        d_act.remainder_(A)
        bact %= A
        base = ctx.wrap_log(d_off, d_act, d_ts, A, max_trace_len=LENGTH)
        new_log, _ = base.append(idx, boff, bact, bts, n_new_traces=n_new)
        torch.cuda.synchronize()
        old = base.declare_counts(K_CAP)
        got, refresh_call, refresh_kern = timed(lambda: (lambda c: (c, c.kernel_ms))(new_log.declare_counts_refresh(base, old, idx)), args.repeats)
        want, full_call, full_kern = timed(lambda: (lambda c: (c, c.kernel_ms))(new_log.declare_counts(K_CAP)), args.repeats)
        parity = bool(np.array_equal(got.packed, want.packed))
        del got, want

        # ceiling log: the listed traces' old versions (touched traces) then their new versions, back to back
        b_act = torch.from_numpy(bact).to(dev)
        old_rows = d_act.view(T, LENGTH)[d_tt]                                                     # k_t x 50
        new_rows = torch.cat((old_rows, b_act[:k_t * 5].view(k_t, 5)), dim=1)                     # k_t x 55
        c_act = torch.cat((old_rows.reshape(-1), new_rows.reshape(-1), b_act[k_t * 5:]))
        del old_rows, new_rows
        c_len = torch.cat((torch.full((k_t,), LENGTH, dtype=torch.int64, device=dev), torch.full((k_t,), LENGTH + 5, dtype=torch.int64, device=dev),
                           torch.full((n_new,), 50, dtype=torch.int64, device=dev)))
        c_off = torch.zeros(len(c_len) + 1, dtype=torch.int64, device=dev)
        torch.cumsum(c_len, 0, out=c_off[1:])
        c_ts = torch.zeros(c_act.numel(), dtype=torch.int64, device=dev)   # K3 reads no timestamp
        ceil_log = ctx.wrap_log(c_off, c_act, c_ts, A, max_trace_len=LENGTH + 5)
        _, _, ceil_kern = timed(lambda: (lambda c: (c, c.kernel_ms))(ceil_log.declare_counts(K_CAP)), args.repeats)
        ceil_log.close()
        ceil_events = int(c_act.numel())
        del c_act, c_len, c_off, c_ts, b_act
        n_vals = len(old.packed)
        src = torch.empty(n_vals, dtype=torch.int64, device=dev)
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
        new_log.close()
        base.close()
        torch.cuda.empty_cache()

        med = lambda v: float(np.median(v))   # noqa: E731
        listed_events = int(boff[-1]) + 2 * LENGTH * k_t   # both versions of the touched traces + the new traces' events
        alg = 4 * listed_events + 8 * k + 3 * 8 * n_vals + 16 * T
        ceiling = med(ceil_kern) + med(cp)
        o = {"kernels": "refresh_check_kernel + max_trace_len_kernel<true> + K3 work-list launches + declare_merge_kernel",
             "traces": T, "events": T * LENGTH, "n_activities": A, "k_cap": K_CAP, "dense_traces": bool(args.dense_traces),
             "listed_traces": k, "touched_traces": k_t, "new_traces": n_new, "batch_events": int(boff[-1]),
             "listed_events_both_logs": listed_events, "count_values": n_vals,
             "refresh_kernel_ms": med(refresh_kern), "refresh_call_ms": med(refresh_call), "refresh_kernel_ms_all": refresh_kern,
             "full_kernel_ms": med(full_kern), "full_call_ms": med(full_call), "full_kernel_ms_all": full_kern,
             "ceiling_count_ms": med(ceil_kern), "ceiling_events": ceil_events, "ceiling_copy_ms": med(cp), "ceiling_ms": ceiling,
             "refresh_over_ceiling": med(refresh_kern) / ceiling, "full_over_refresh": med(full_kern) / med(refresh_kern),
             "refresh_algorithmic_bytes": alg, "refresh_algorithmic_GBps": alg / (med(refresh_kern) * 1e-3) / 1e9,
             "parity_refresh_equals_full": parity, "gpu": name, "power_limit": power}
        print(json.dumps(o), flush=True)
        lines.append(o)
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            for o in lines:
                f.write(json.dumps(o) + "\n")


if __name__ == "__main__":
    main()
