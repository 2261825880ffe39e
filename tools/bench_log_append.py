"""Growing a resident log (siesta_log_append, csrc/append.cu): one JSON line per size.

Full size: the base is the flagship's 100 M traces x 50 events (bench.make_log_device, generated on the GPU, 60.8 GB); the
batch touches 1 M existing traces with 5 events each and adds 1 M new traces of 50 events.  Reported: kernel time
(CUDA events inside the call) and call time (host clock; the call ends in a stream synchronise), algorithmic GB/s against
the measured HBM peak and the 7.7 TB/s data sheet, a torch copy_ of about the same byte count timed in the same run
(the in-run ceiling), and the host -> device time of the batch.  Reload comparison (--reload-traces, default 10 M): the
same append next to a full siesta_log_load of the merged log from pinned host memory.  Dense (--dense-traces, default
10 M): a batch that touches every trace with 5 events, so pieces hold ~50 events instead of ~5 000.  Parity at every
size: sampled traces (touched, new, untouched, first and last) read back with siesta_log_read equal the base tensors +
the batch.
`python tools/bench_log_append.py [--traces N] [--reload-traces N] [--dense-traces N] [--sample N]`"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from sequencedetectionqueryexecutor_b200 import api  # noqa: E402
from sequencedetectionqueryexecutor_b200._lib import check, lib  # noqa: E402

LENGTH, N_ACT, SEED, GAP_S = 50, 20, 0x51E57A05, 600
DATASHEET_GBS = 7700.0


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:   # the number is still printed, without its power limit
        out = f"unknown ({e})"
    return name, out


def make_batch(torch, d_ts, T, touched, touched_len, new, new_len, seed):
    """Touched traces (ascending, distinct) get `touched_len` events after their last one; new traces get `new_len`."""
    rng = np.random.default_rng(seed)
    tt = np.sort(rng.choice(T, size=touched, replace=False)).astype(np.int64)
    last = d_ts[torch.from_numpy(tt * LENGTH + LENGTH - 1).to(d_ts.device)].cpu().numpy()
    idx = np.concatenate((tt, T + np.arange(new, dtype=np.int64)))
    lens = np.concatenate((np.full(touched, touched_len), np.full(new, new_len))).astype(np.int64)
    off = np.zeros(len(idx) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    act = rng.integers(0, N_ACT, size=int(off[-1]), dtype=np.int32)
    gaps = rng.integers(1, GAP_S + 1, size=int(off[-1]), dtype=np.int64) * 1000
    start = np.concatenate((last, 1577836800000 + rng.integers(0, 30 * 86400, size=new, dtype=np.int64) * 1000))
    seg_start = np.repeat(off[:-1], lens)
    cs = np.cumsum(gaps)
    ts = cs - np.concatenate(([0], cs))[seg_start] + np.repeat(start, lens)
    return idx, off, act, ts


def parity(torch, log, d_act, d_ts, T, idx, off, act, ts, n_sample, seed):
    """siesta_log_read of sampled traces == base tensors + batch (the base is fixed-length: trace t = [t*50, t*50+50))."""
    rng = np.random.default_rng(seed)
    T2 = log.n_traces
    k_touched = int(np.searchsorted(idx, T))
    pick = [np.arange(min(5, T2)), np.arange(max(T2 - 5, 0), T2), rng.choice(idx[:k_touched], size=min(n_sample // 3, k_touched), replace=False)
            if k_touched else np.zeros(0, np.int64), rng.choice(idx[k_touched:], size=min(n_sample // 3, len(idx) - k_touched), replace=False)
            if len(idx) > k_touched else np.zeros(0, np.int64)]
    pick.append(rng.integers(0, T, size=max(n_sample - sum(len(p) for p in pick), 0)))
    sample = np.unique(np.concatenate(pick).astype(np.int64))
    base_rows = sample[sample < T]
    g = torch.from_numpy((base_rows[:, None] * LENGTH + np.arange(LENGTH)[None, :]).reshape(-1)).to(d_act.device)
    b_act = d_act[g].cpu().numpy().reshape(-1, LENGTH)
    b_ts = d_ts[g].cpu().numpy().reshape(-1, LENGTH)
    row_of = {int(t): r for r, t in enumerate(base_rows)}
    pos_of = {int(t): i for i, t in enumerate(idx)}
    o = np.zeros(2, dtype=np.int64)
    ok = True
    for t in sample:
        t = int(t)
        want_a, want_t = [], []
        if t in row_of:
            want_a.append(b_act[row_of[t]])
            want_t.append(b_ts[row_of[t]])
        if t in pos_of:
            i = pos_of[t]
            want_a.append(act[off[i]:off[i + 1]])
            want_t.append(ts[off[i]:off[i + 1]])
        wa = np.concatenate(want_a) if want_a else np.zeros(0, np.int32)
        wt = np.concatenate(want_t) if want_t else np.zeros(0, np.int64)
        ga = np.zeros(max(len(wa), 1), dtype=np.int32)
        gt = np.zeros(max(len(wa), 1), dtype=np.int64)
        check(lib().siesta_log_read(log._h, t, t + 1, api._ptr(o), None, None))
        if o[1] - o[0] != len(wa):
            ok = False
            break
        check(lib().siesta_log_read(log._h, t, t + 1, api._ptr(o), api._ptr(ga), api._ptr(gt)))
        if not (np.array_equal(ga[:len(wa)], wa) and np.array_equal(gt[:len(wa)], wt)):
            ok = False
            break
    return ok, len(sample)


def alg_bytes(T, E, k, NB, n_new):
    """12 B/event + 8 B/trace read from the old log, 12 B/event of the batch + 16 B per listed trace, 12 B/event +
    8 B/trace written."""
    return 12 * E + 8 * (T + 1) + 12 * NB + 16 * k + 12 * (E + NB) + 8 * (T + n_new + 1)


def run_size(torch, ctx, T, touched, new, repeats, n_sample, reload_cmp):
    dev = torch.device("cuda", 0)
    d_off, d_act, d_ts = bench.make_log_device(torch, dev, 0, T, T, LENGTH, N_ACT, SEED, GAP_S)
    base = ctx.wrap_log(d_off, d_act, d_ts, N_ACT, max_trace_len=LENGTH)
    idx, off, act, ts = make_batch(torch, d_ts, T, touched, 5, new, 50, seed=T)
    E, k, NB = T * LENGTH, len(idx), int(off[-1])
    torch.cuda.synchronize()
    kern, call = [], []   # --repeats calls after one warm-up; min and median are reported
    new_log = None
    for r in range(repeats + 1):   # the first call is the warm-up
        if new_log is not None:
            new_log.close()
        t0 = time.perf_counter()
        new_log, ms = base.append(idx, off, act, ts, n_new_traces=new)
        dt = (time.perf_counter() - t0) * 1e3
        if r:
            kern.append(ms)
            call.append(dt)
    ok, n_checked = parity(torch, new_log, d_act, d_ts, T, idx, off, act, ts, n_sample, seed=T + 1)
    # host -> device time of the batch (pageable numpy, as the call takes it)
    t0 = time.perf_counter()
    for x in (idx, off, act, ts):
        torch.from_numpy(x).to(dev)
    torch.cuda.synchronize()
    h2d_ms = (time.perf_counter() - t0) * 1e3
    out = {}
    if reload_cmp:
        # the merged log on the host in pinned memory, then a full siesta_log_load of it
        T2, E2 = new_log.n_traces, new_log.n_events
        h_off = torch.empty(T2 + 1, dtype=torch.int64, pin_memory=True).numpy()
        h_act = torch.empty(E2, dtype=torch.int32, pin_memory=True).numpy()
        h_ts = torch.empty(E2, dtype=torch.int64, pin_memory=True).numpy()
        check(lib().siesta_log_read(new_log._h, 0, T2, api._ptr(h_off), api._ptr(h_act), api._ptr(h_ts)))
        new_log.close()
        new_log = None
        loads = []
        for _ in range(2):
            t0 = time.perf_counter()
            fresh = ctx.load_log(h_off, h_act, h_ts, N_ACT)
            loads.append((time.perf_counter() - t0) * 1e3)
            fresh.close()
        out["reload_full_load_ms"] = min(loads)
        out["reload_full_load_ms_all"] = loads
        out["reload_over_append_call_median"] = min(loads) / float(np.median(call))
        del h_off, h_act, h_ts
    if new_log is not None:
        new_log.close()
    base.close()
    # in-run ceiling: torch copy_ of the base columns (read + write ~ the algorithmic byte count), rescaled to it exactly
    dst_a, dst_t = torch.empty_like(d_act), torch.empty_like(d_ts)
    cp = []
    for r in range(repeats + 1):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        dst_a.copy_(d_act)
        dst_t.copy_(d_ts)
        s1.record()
        torch.cuda.synchronize()
        if r:
            cp.append(s0.elapsed_time(s1))
    copy_bytes = 2 * (d_act.numel() * 4 + d_ts.numel() * 8)
    del dst_a, dst_t, d_off, d_act, d_ts
    torch.cuda.empty_cache()
    a_bytes = alg_bytes(T, E, k, NB, new)
    kms = min(kern)
    copy_equiv_ms = min(cp) * a_bytes / copy_bytes
    peak, peak_src = bench.measured_peak_gbs()
    gbs = a_bytes / (kms * 1e-3) / 1e9
    out.update({"kernel": "ap_offsets_kernel + ap_copy_kernel", "traces": T, "events": E, "listed_traces": k, "touched_traces": touched,
                "new_traces": new, "batch_events": NB, "kernel_ms": kms, "kernel_ms_all": kern, "call_ms": min(call), "call_ms_median": float(np.median(call)), "call_ms_all": call,
                "algorithmic_bytes": a_bytes, "algorithmic_GBps": gbs, "frac_of_measured_hbm_peak": gbs / peak, "measured_peak_GBps": peak,
                "measured_peak_source": peak_src, "frac_of_datasheet_7700": gbs / DATASHEET_GBS, "copy_ms": min(cp), "copy_bytes": copy_bytes,
                "copy_ms_at_algorithmic_bytes": copy_equiv_ms, "kernel_over_copy": kms / copy_equiv_ms, "batch_h2d_ms": h2d_ms,
                "parity": bool(ok), "parity_traces_checked": n_checked})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--traces", type=int, default=100_000_000)
    ap.add_argument("--touched", type=int, default=1_000_000)
    ap.add_argument("--new", type=int, default=1_000_000)
    ap.add_argument("--reload-traces", type=int, default=10_000_000)
    ap.add_argument("--dense-traces", type=int, default=10_000_000, help="a batch that touches every trace (0: skip)")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--sample", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_log_append: no CUDA device")
    name, power = card()
    ctx = api.Context(0)
    sizes = [("full", args.traces, args.touched, args.new, False)]
    if args.reload_traces:
        f = args.reload_traces / args.traces
        sizes.append(("reload comparison", args.reload_traces, max(int(args.touched * f), 1), max(int(args.new * f), 1), True))
    if args.dense_traces:   # every trace touched: pieces of ~50 old + 5 new events instead of ~5 000
        sizes.append(("dense, every trace touched", args.dense_traces, args.dense_traces, 0, False))
    for label, T, touched, new, reload_cmp in sizes:
        res = run_size(torch, ctx, T, touched, new, args.repeats, args.sample, reload_cmp)
        res.update({"size": label, "gpu": name, "power_limit": power})
        print(json.dumps(res), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
