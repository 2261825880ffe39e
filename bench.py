#!/usr/bin/env python
"""bench.py — events scanned/sec of the /detection verification path on B200.

Default workload = BASELINE.json configs[4], the configuration the metric is quoted on: the 6-event pattern with ||, !
and gap constraints over a 100 M-trace x 50-event log (60.8 GB CSR), STRONG scaling: the same log at every N, each rank
holding 100 M / N traces (QueryPlanPatternDetection.execute, J/model/Queries/QueryPlans/Detection/
QueryPlanPatternDetection.java:106-131, stands behind it in the reference).

  python bench.py --gpus N --steps K --warmup W            # the CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's result to DIR/<name>.npy

A step = one /detection request (SaseConnector.evaluate + clearOccurrences == siesta_detect) over the whole log; at
N > 1 it ends when EVERY rank holds the joined, decoded match list of all ranks (siesta_exchange_*: the device-side
all-gather of the compact result blocks over NVLink).  `value` has the log resident in HBM; `e2e` goes through the
host-buffer C-ABI call (siesta_evaluate_events) on a host-resident slice of the log with the host<->device copies inside
the timed region.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the bench writes nothing into the source tree, which may be read-only

from sequencedetectionqueryexecutor_b200 import _abi as abi  # noqa: E402

GAP6 = [dict(kind=abi.STATE_NORMAL, types=[0]),
        dict(kind=abi.STATE_OR, types=[1, 2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 10)]),
        dict(kind=abi.STATE_NEGATIVE, types=[3]), dict(kind=abi.STATE_NORMAL, types=[4]),
        dict(kind=abi.STATE_NORMAL, types=[5], preds=[(abi.ATTR_POSITION, abi.OP_GE, 3, 2)])]
GAP6_TEXT = "a (b|c) !d e f; gap within 10 (0,1), gap atleast 2 (3,4) (EventTs route, returnAll=false)"
NKP = "detect_nkp_kernel<NPL=3, rank space> (K1-P: table-driven class planes on the FMA pipe + window walks, one lane per trace)"

WORKLOADS = {
    # BASELINE.json configs[4] (SURVEY.md §8(d) cfg 5): 100M traces x 50 events, 20 activities, gaps U{1..600} s
    "detection_gap6_100Mx50": dict(n_traces=100_000_000, min_len=50, max_len=50, n_act=20, max_gap_s=600, seed=0x51E57A05,
                                   bytes_per_event=4, pattern=GAP6_TEXT, kernel=NKP, states=GAP6, e2e_traces=4_000_000),
    # the same query on 4M traces (profiles/, quick A/B runs)
    "detection_gap6_4Mx50": dict(n_traces=4_000_000, min_len=50, max_len=50, n_act=20, max_gap_s=600, seed=0x51E57A05,
                                 bytes_per_event=4, pattern=GAP6_TEXT, kernel=NKP, states=GAP6, e2e_traces=4_000_000),
    # the same query with returnAll=true: what the JNI drop-in asks for (the seam does not carry returnAll: INTEGRATION.md 1)
    "detection_gap6_all_4Mx50": dict(n_traces=4_000_000, min_len=50, max_len=50, n_act=20, max_gap_s=600, seed=0x51E57A05,
                                     bytes_per_event=4, pattern=GAP6_TEXT.replace("returnAll=false", "returnAll=true"),
                                     kernel=NKP + "; traces with more than one engine match re-run on the staged kernel, which reads their timestamps for the overlap test",
                                     flags=abi.F_RETURN_ALL, states=GAP6, e2e_traces=4_000_000),
    # BASELINE.json configs[1]: /detection Kleene pattern a+ b* with a within-10-minutes time constraint,
    # 1M traces x 100 events (20 activity types, gaps U{1..120} s).  SURVEY.md §8(d) cfg 2.
    "detection_kleene_1Mx100": dict(n_traces=1_000_000, min_len=100, max_len=100, n_act=20, max_gap_s=120, seed=0x51E57A02,
                                    bytes_per_event=12, pattern="a+ b* within 10 minutes (EventTs route, returnAll=false)",
                                    kernel="detect_kernel<W=1, FAST_FK2> (K1: filter + a+ b* closed form + staged output)",
                                    states=[dict(kind=abi.STATE_KLEENE_PLUS, types=[0]),
                                            dict(kind=abi.STATE_KLEENE_STAR, types=[1],
                                                 preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], e2e_traces=1_000_000),
    # Kleene patterns outside the a+ b* closed form (VERDICT r1 item 6): a b+ c has its own closed form since round 2
    # (class NP1), also with constraints that reference states before the `+` state
    "detection_abc_kleene_1Mx100": dict(n_traces=1_000_000, min_len=100, max_len=100, n_act=20, max_gap_s=120, seed=0x51E57A02,
                                        bytes_per_event=4, pattern="a b+ c (EventTs route, returnAll=false)",
                                        kernel="detect_kernel<W=1, FAST_NP1> (K1: filter + one-`+`-state closed form + staged output)",
                                        states=[dict(kind=abi.STATE_NORMAL, types=[0]), dict(kind=abi.STATE_KLEENE_PLUS, types=[1]),
                                                dict(kind=abi.STATE_NORMAL, types=[2])], e2e_traces=1_000_000),
    "detection_abc_kleene_gap_1Mx100": dict(n_traces=1_000_000, min_len=100, max_len=100, n_act=20, max_gap_s=120, seed=0x51E57A02,
                                            bytes_per_event=4, pattern="a b+ c, gap within 20 (0,2) (EventTs route, returnAll=false)",
                                            kernel="detect_kernel<W=1, FAST_NP1> (K1: filter + one-`+`-state closed form, every start on its filtered masks)",
                                            states=[dict(kind=abi.STATE_NORMAL, types=[0]), dict(kind=abi.STATE_KLEENE_PLUS, types=[1]),
                                                    dict(kind=abi.STATE_NORMAL, types=[2], preds=[(abi.ATTR_POSITION, abi.OP_LE, 0, 20)])],
                                            e2e_traces=1_000_000),
    # the reference's own Kleene test shape (EvaluateComplexQueries.java:101-103): one `*` state, no constraints
    "detection_abstar_c_1Mx100": dict(n_traces=1_000_000, min_len=100, max_len=100, n_act=20, max_gap_s=120, seed=0x51E57A02,
                                      bytes_per_event=4, pattern="a b* c (EventTs route, returnAll=false)",
                                      kernel="detect_kernel<W=1, FAST_NP1> (K1: filter + one-Kleene-state closed form + staged output)",
                                      states=[dict(kind=abi.STATE_NORMAL, types=[0]), dict(kind=abi.STATE_KLEENE_STAR, types=[1]),
                                              dict(kind=abi.STATE_NORMAL, types=[2])], e2e_traces=1_000_000),
    "detection_kleene_all_1Mx100": dict(n_traces=1_000_000, min_len=100, max_len=100, n_act=20, max_gap_s=120, seed=0x51E57A02,
                                        bytes_per_event=12, pattern="a+ b* within 10 minutes, returnAll=true",
                                        kernel="detect_kernel<FAST_NONE> (K1: filter + run-list engine)", flags=abi.F_RETURN_ALL,
                                        states=[dict(kind=abi.STATE_KLEENE_PLUS, types=[0]),
                                                dict(kind=abi.STATE_KLEENE_STAR, types=[1],
                                                     preds=[(abi.ATTR_TIMESTAMP, abi.OP_LE, 0, 600)])], e2e_traces=1_000_000),
    # configs[0] shape: A_ B_ on 10k traces x ~40 events (no constraint: 4 B/event).
    "detection_ab_10kx40": dict(n_traces=10_000, min_len=30, max_len=50, n_act=20, max_gap_s=600, seed=0x51E57A01,
                                bytes_per_event=4, pattern="A_ B_ (EventTs route, returnAll=false)",
                                kernel="detect_nkp_kernel<NPL=2, rank space>",
                                states=[dict(kind=abi.STATE_NORMAL, types=[0]), dict(kind=abi.STATE_NORMAL, types=[1])],
                                e2e_traces=10_000),
}
DEFAULT_WORKLOAD = "detection_gap6_100Mx50"
CHUNK = 1_250_000      # traces per generator chunk: 100 M / 8 GPUs = 10 chunks, so every shard boundary is a chunk boundary
SAMPLE_TRACES = 1_000_000   # the CPU arms (cpu_baseline, --impl reference) run the first SAMPLE_TRACES traces of the log
DUMP_BYTES = 64_000_000     # --dump-outputs writes at most this many bytes in all
DUMP_SEED = 0x51E57A00


def dump_outputs(dm, device_index, out_dir):
    """--dump-outputs: the columns a caller of the timed path receives (DeviceMatches.tensors(): matching trace ids, the
    occurrence and event offsets, the event columns, the error and unsupported trace lists) as DIR/<column>.npy, and the
    result sizes as DIR/sizes.npy.  An empty column (usually the error and unsupported lists) is not written: its length,
    zero, is in sizes.npy.  float64 holds every value exactly (ids, offsets, positions and millisecond timestamps are
    integers below 2**53).  A column longer than its share of DUMP_BYTES is written at a sorted sample of positions
    drawn from (DUMP_SEED, its length), so two builds that compute the same result write the same files."""
    import torch
    cols = {k: t for k, t in dm.tensors(device_index).items() if t.numel()}
    cap = (DUMP_BYTES - 4096 * (len(cols) + 1)) // (8 * max(len(cols), 1))   # 4096: room for each file's .npy header
    os.makedirs(out_dir, exist_ok=True)
    sizes = [dm.n_traces, dm.n_occurrences, dm.n_events, dm.n_matches_emitted, dm.n_ref_errors, dm.n_unsupported]
    np.save(os.path.join(out_dir, "sizes.npy"), np.array(sizes, dtype=np.float64))
    sampled = {}
    for name, t in sorted(cols.items()):
        n = t.numel()
        if n > cap:
            at = np.sort(np.random.default_rng([DUMP_SEED, n]).choice(n, cap, replace=False))
            t = t[torch.from_numpy(at).to(t.device)]
            sampled[name] = f"{cap} of {n}"
        np.save(os.path.join(out_dir, f"{name}.npy"), t.to(torch.float64).cpu().numpy())
    print(f"bench.py: wrote {len(cols) + 1} arrays to {out_dir}" + (f"; sampled: {sampled}" if sampled else ""),
          file=sys.stderr, flush=True)


def full_size_properties(log, nfa, flags, states, d_off, d_act, d_ts, device_index):
    """Checks on EVERY occurrence of the full-size result, on the device with torch (the CPU oracle sees a sample only):
    trace ids strictly ascending, CSR offsets consistent, positions strictly increasing inside an occurrence, every
    reported event is the log's event at (trace, position) - activity and, on the EventTs route, a timestamp at most a
    second below the log's (SaseEvent.getEventBoth rebuilds it from whole seconds) - and, for patterns without a Kleene state asked for the
    first-largest occurrence, one occurrence per trace with one event per positive state, of that state's types, that
    satisfies the state's position predicates.  Returns {name: bool}."""
    import torch
    dm = log.detect_device(nfa, flags=flags)
    t = dm.tensors(device_index)
    out = {}
    n_tr, n_occ, n_ev = dm.n_traces, dm.n_occurrences, dm.n_events
    tr, occ_off, ev_off, pos = t["trace_idx"], t["occ_off"], t["ev_off"], t["ev_pos"].long()
    out["trace_ids_ascending"] = bool(n_tr < 2 or torch.all(tr[1:] > tr[:-1]).item())
    out["offsets_consistent"] = bool(occ_off[0].item() == 0 and occ_off[-1].item() == n_occ and ev_off[0].item() == 0 and
                                     ev_off[-1].item() == n_ev and torch.all(occ_off[1:] > occ_off[:-1]).item() and
                                     torch.all(ev_off[1:] > ev_off[:-1]).item())
    first = torch.zeros(n_ev, dtype=torch.bool, device=pos.device)
    first[ev_off[:-1]] = True
    out["positions_increase_inside_occurrences"] = bool(torch.all((pos[1:] > pos[:-1]) | first[1:]).item())
    # the trace of every event: occurrence of the event -> trace of the occurrence
    occ_of_ev = torch.repeat_interleave(torch.arange(n_occ, device=pos.device), ev_off[1:] - ev_off[:-1])
    tr_of_occ = torch.repeat_interleave(tr, occ_off[1:] - occ_off[:-1])
    at = d_off[tr_of_occ[occ_of_ev]] + pos
    out["events_are_the_logs_events"] = bool(torch.all(pos < (d_off[tr_of_occ[occ_of_ev] + 1] - d_off[tr_of_occ[occ_of_ev]])).item() and
                                             torch.all(t["ev_act"] == d_act[at]).item())
    if not (flags & abi.F_EVT_POS):
        dts = d_ts[at] - t["ev_ts_ms"]           # SaseEvent.getEventBoth: whole seconds after the first filtered event
        out["timestamps_within_a_second_of_the_logs"] = bool(torch.all((dts >= 0) & (dts < 1000)).item())
    positive = [s for s in states if s["kind"] != abi.STATE_NEGATIVE]
    if not (flags & abi.F_RETURN_ALL) and all(s["kind"] in (abi.STATE_NORMAL, abi.STATE_OR, abi.STATE_NEGATIVE) for s in states):
        k = len(positive)
        uniform = n_occ == n_tr and n_ev == k * n_occ and bool(torch.all(ev_off == k * torch.arange(n_occ + 1, device=pos.device)).item())
        out["one_occurrence_of_k_events_per_trace"] = uniform
        if uniform:
            act_m, rank_m = t["ev_act"].view(n_occ, k), t["ev_rank"].view(n_occ, k)
            ord_of = {}
            for i, s_ in enumerate(states):
                if s_["kind"] != abi.STATE_NEGATIVE:
                    ord_of[i] = len(ord_of)
            types_ok, preds_ok = True, True
            for i, s_ in enumerate(states):
                if i not in ord_of:
                    continue
                col = act_m[:, ord_of[i]]
                types_ok &= bool(torch.isin(col, torch.tensor(s_["types"], device=col.device, dtype=col.dtype)).all().item())
                for (attr, op, ref, c) in s_.get("preds", []):
                    if attr != abi.ATTR_POSITION or (flags & abi.F_EVT_POS):
                        continue             # EventTs route: `position` is the index in the filtered list = ev_rank
                    lhs, rhs = rank_m[:, ord_of[i]], rank_m[:, ord_of[ref]] + c
                    preds_ok &= bool(((lhs <= rhs) if op == abi.OP_LE else (lhs >= rhs)).all().item())
            out["events_have_their_states_types"] = types_ok
            out["position_predicates_hold"] = preds_ok
    out["occurrences_checked"] = int(n_occ)
    dm.close()
    return out


def make_log_fast(n_traces, min_len, max_len, n_act, seed, max_gap_s, rank=0):
    """Host generator (variable-length workloads); same distribution as tests/gen.make_log, vectorised."""
    rng = np.random.default_rng([seed, rank])
    if min_len == max_len:
        lens = np.full(n_traces, min_len, dtype=np.int64)
    else:
        lens = rng.integers(min_len, max_len + 1, size=n_traces, dtype=np.int64)
    off = np.zeros(n_traces + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    E = int(off[-1])
    act = rng.integers(0, n_act, size=E, dtype=np.int32)
    ts = rng.integers(1, max_gap_s + 1, size=E, dtype=np.int64)
    ts *= 1000
    np.cumsum(ts, out=ts)
    start = 1577836800000 + rng.integers(0, 30 * 86400, size=n_traces, dtype=np.int64) * 1000
    first = np.minimum(off[:-1], max(E - 1, 0))
    shift = start - ts[first]
    ts += np.repeat(shift, lens)
    return off, act, ts


def make_log_device(torch, dev, t_begin, t_end, n_total, length, n_act, seed, max_gap_s, ranges=None):
    """Traces [t_begin, t_end) - or the trace ranges `ranges` back to back (a block-cyclic shard) - of the fixed-length
    synthetic log, generated on the GPU (the 100 M-trace log is 60.8 GB: it never exists on the host).  The generator is
    keyed by (seed, chunk of CHUNK traces), so a shard holds exactly the traces the one-GPU run holds at the same global
    indices, whatever N and the block layout are."""
    if ranges is None:
        ranges = [(t_begin, t_end)]
    n = sum(hi - lo for lo, hi in ranges)
    E = n * length
    off = torch.arange(0, E + 1, length, dtype=torch.int64, device=dev)
    act = torch.empty(E, dtype=torch.int32, device=dev)
    ts = torch.empty(E, dtype=torch.int64, device=dev)
    g = torch.Generator(device=dev)
    at = 0   # local index of the range's first trace
    for r_lo, r_hi in ranges:
        for c in range(r_lo // CHUNK, (r_hi + CHUNK - 1) // CHUNK):
            c0, c1 = c * CHUNK, min(n_total, (c + 1) * CHUNK)
            m = c1 - c0
            g.manual_seed(int(seed) * 1000003 + c)
            a = torch.randint(0, n_act, (m * length,), dtype=torch.int32, device=dev, generator=g)
            gaps = torch.randint(1, max_gap_s + 1, (m, length), dtype=torch.int64, device=dev, generator=g)
            gaps *= 1000
            torch.cumsum(gaps, dim=1, out=gaps)
            start = 1577836800000 + torch.randint(0, 30 * 86400, (m, 1), dtype=torch.int64, device=dev, generator=g) * 1000
            gaps += start
            lo, hi = max(c0, r_lo), min(c1, r_hi)     # the part of the chunk this range owns
            d0 = at + (lo - r_lo)
            act[d0 * length:(d0 + hi - lo) * length] = a[(lo - c0) * length:(hi - c0) * length]
            ts[d0 * length:(d0 + hi - lo) * length] = gaps.view(-1)[(lo - c0) * length:(hi - c0) * length]
            del a, gaps, start
        at += r_hi - r_lo
    return off, act, ts


class ClockSampler:
    """SM clock, power and throttle reasons of this rank's GPU sampled DURING the timed region (B200_PROFILING.md), through
    NVML inside the process (a thread polling every 20 ms).  Spawning `nvidia-smi -lms` per rank instead initialises NVML
    in eight new processes right when the timed steps start and stalls driver calls for ~200 ms (measured on the 8-GPU
    box: p50 4.3 ms, p99 219 ms per request); nvidia-smi remains the fallback when the NVML binding is missing."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()
        self.mode = None
        self.proc = None
        self.marks = [0, None]

    def start(self):
        if os.environ.get("SIESTA_BENCH_NO_SAMPLER"):   # diagnosis only: is a hiccup the sampler's?
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            try:
                q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                              "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.mode = "smi"
                self.t = threading.Thread(target=self._read, daemon=True)
                self.t.start()
            except Exception:
                self.mode = None

    def _poll(self):
        nv = self.nv
        R = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
             "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        pw, k = 0.0, 0
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if k % 8 == 0 and not os.environ.get("SIESTA_BENCH_NO_POWER"):   # the power read goes to the board's controller: slower, rarer
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                k += 1
                self.samples.append((sm, self.max_sm, pw, {k2 for k2, v in R.items() if bits & v}))
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                self.samples.append((float(f[1]), float(f[2]), float(f[3]),
                                     {n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8])
                                      if v.lower().startswith("active")}))
            except (ValueError, IndexError):
                continue

    def mark_begin(self):
        """Samples before this point (warm-up) are not reported."""
        self.marks[0] = len(self.samples)

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML binding and no nvidia-smi"]}
        time.sleep(0.05)
        self.stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()
        got = self.samples[self.marks[0]:] or self.samples[-3:]
        sm = [x[0] for x in got]
        reasons = set().union(*[x[3] for x in got]) if got else set()
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(x[1] for x in got) if got else None,
                "power_w_max": max(x[2] for x in got) if got else None, "reasons": sorted(reasons), "samples": len(got),
                "source": "NVML in-process, 20 ms" if self.mode == "nvml" else "nvidia-smi -lms 100"}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_bytes(workload, traces):
    """DRAM bytes (read + write) of one K1 launch from the committed ncu --set full capture (profiles/k1_traffic.json:
    bytes per trace of this query, measured at a full launch), scaled to this launch; None if absent."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))
        d = d.get(workload) or d[{"detection_gap6_100Mx50": "detection_gap6_4Mx50"}[workload]]
        return int(d["dram_bytes_per_trace"] * traces), d.get("capture", "committed ncu capture")
    except Exception:
        return None, None


def config_of(args, wl):
    """The `config` object: identical in both arms (the driver compares them)."""
    return {"workload": args.workload, "pattern": wl["pattern"], "traces": wl["n_traces"],
            "events": wl["n_traces"] * wl["min_len"] if wl["min_len"] == wl["max_len"] else None,
            "activities": wl["n_act"],
            "cpu_sample": f"first {min(SAMPLE_TRACES, wl['n_traces'])} traces of the log"}


def sample_log(wl):
    """The first SAMPLE_TRACES traces of the workload's log on the host, for the CPU arms.  Fixed-length workloads take
    them from the device generator (a GPU is needed to reproduce the exact bits); without one the host generator draws
    a log of the same distribution."""
    ns = min(SAMPLE_TRACES, wl["n_traces"])
    if wl["min_len"] == wl["max_len"]:
        try:
            import torch
            if torch.cuda.is_available():
                dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
                o, a, t = make_log_device(torch, dev, 0, ns, wl["n_traces"], wl["min_len"], wl["n_act"], wl["seed"], wl["max_gap_s"])
                out = o.cpu().numpy(), a.cpu().numpy(), t.cpu().numpy()
                del o, a, t
                torch.cuda.empty_cache()
                return out, "device generator (same bits as the GPU arm)"
        except Exception:
            pass
        return make_log_fast(ns, wl["min_len"], wl["max_len"], wl["n_act"], wl["seed"], wl["max_gap_s"]), "host generator (same distribution)"
    off, act, ts = make_log_fast(wl["n_traces"], wl["min_len"], wl["max_len"], wl["n_act"], wl["seed"], wl["max_gap_s"])
    e = int(off[ns])
    return (off[:ns + 1], act[:e], ts[:e]), "host generator (same bits as the GPU arm)"


def run_reference(args, wl, world, rank, emit):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port; the Java original
    cannot run here: no JVM) on all host threads; each step = the first SAMPLE_TRACES traces of the workload's log,
    the same sample the GPU arm's cpu_baseline and parity check use."""
    if rank != 0:
        return
    nfa = abi.make_nfa(wl["states"])
    flags = wl.get("flags", 0)
    threads = os.cpu_count() or 1
    (off, act, ts), how = sample_log(wl)
    import oracle
    for _ in range(args.warmup):
        oracle.detect(off, act, ts, nfa, flags=flags, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle.detect(off, act, ts, nfa, flags=flags, n_threads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    v = len(act) / dt
    sample = f"first {len(off) - 1} traces ({len(act)} events) of the log per step; {how}"
    emit({
        "impl": "reference", "metric": "events scanned/sec (/detection verification)", "value": v, "unit": "events/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config_of(args, wl),
        "cpu_baseline": {"value": v, "unit": "events/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def main():
    # stdout carries exactly ONE JSON line: anything a library prints there while the bench runs (NCCL's version banner,
    # for one) is sent to stderr instead
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--traces", type=int, default=0, help="override the log's trace count (debugging; invalidates the metric)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-properties", action="store_true", help="skip the size-independent checks of the full result")
    ap.add_argument("--e2e-extra-flags", type=int, default=0,
                    help="experiment: OR these SIESTA_F_* bits into the e2e leg's request (16 = no event columns: ev_pos only)")
    ap.add_argument("--e2e-int32", action="store_true", help="e2e leg through the int32 activity column only (siesta_evaluate_events)")
    ap.add_argument("--blocks", type=int, default=1,
                    help="N > 1: blocks per shard of the block-cyclic layout (siesta_log_set_blocks: block b is pulled and decoded "
                         "while block b + 1 is scanned).  Default 1 = contiguous shards: measured faster on 2 and 8 B200 "
                         "(profiles/r02b_exchange_blocks.md)")
    ap.add_argument("--join", default="allgather", choices=["allgather", "none"],
                    help="N > 1: allgather = every rank ends the step with the decoded match list of all ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step as DIR/<column>.npy (float64, at most 64 MB in all; "
                         "a seeded sample of a longer column) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    wl = dict(WORKLOADS[args.workload])
    if args.traces:
        wl["n_traces"] = args.traces
        wl["e2e_traces"] = min(wl["e2e_traces"], args.traces)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's result (--impl b200)")
    if args.dump_outputs and world > 1 and args.join != "allgather":
        ap.error("--dump-outputs at N > 1 needs --join allgather: without it no rank holds the whole result")

    if args.impl == "reference":
        run_reference(args, wl, world, rank, emit)
        return

    import torch
    import torch.distributed as dist

    from sequencedetectionqueryexecutor_b200 import api
    from sequencedetectionqueryexecutor_b200 import distributed as D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- this rank's shard of the log: contiguous trace range [t_lo, t_hi) (strong scaling: the log is fixed)
    nfa = abi.make_nfa(wl["states"])
    flags = wl.get("flags", 0)
    fixed = wl["min_len"] == wl["max_len"]
    NT = wl["n_traces"]
    blocks = None     # block-cyclic shard: [(global first, global end)] of this rank's blocks
    if fixed and world > 1 and args.join == "allgather" and args.blocks > 1:
        # Block-cyclic shards (siesta_log_set_blocks): the log is cut into blocks * world blocks of consecutive traces, rank
        # r holds blocks r, world + r, ...: block b + 1 is scanned while block b of every rank is pulled and decoded.
        nb = args.blocks * world
        bounds = [(NT * i) // nb for i in range(nb + 1)]
        if NT >= nb * CHUNK:
            bounds = [min(NT, -(-b // CHUNK) * CHUNK) for b in bounds]     # block boundaries on generator chunks
        blocks = [(bounds[c * world + rank], bounds[c * world + rank + 1]) for c in range(args.blocks)]
        t_lo, t_hi = blocks[0]
        d_off, d_act, d_ts = make_log_device(torch, dev, 0, 0, NT, wl["min_len"], wl["n_act"], wl["seed"], wl["max_gap_s"], ranges=blocks)
    elif fixed:
        per = -(-NT // world)
        per = -(-per // CHUNK) * CHUNK if NT >= world * CHUNK else per     # shard boundaries on generator chunks
        t_lo, t_hi = min(NT, rank * per), min(NT, (rank + 1) * per)
        d_off, d_act, d_ts = make_log_device(torch, dev, t_lo, t_hi, NT, wl["min_len"], wl["n_act"], wl["seed"], wl["max_gap_s"])
    else:
        g_off, g_act, g_ts = make_log_fast(NT, wl["min_len"], wl["max_len"], wl["n_act"], wl["seed"], wl["max_gap_s"])
        b = D.shard_bounds(g_off, world)
        t_lo, t_hi = int(b[rank]), int(b[rank + 1])
        e0, e1 = int(g_off[t_lo]), int(g_off[t_hi])
        d_off = torch.from_numpy(g_off[t_lo:t_hi + 1] - e0).to(dev)
        d_act = torch.from_numpy(g_act[e0:e1]).to(dev)
        d_ts = torch.from_numpy(g_ts[e0:e1]).to(dev)
    T, E = d_off.numel() - 1, d_act.numel()
    E_total = torch.tensor([E], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(E_total)
    E_total = int(E_total.item())

    ctx = api.Context(local_rank)
    log = ctx.wrap_log(d_off, d_act, d_ts, wl["n_act"], max_trace_len=wl["max_len"])
    log.set_first_trace(t_lo)
    if blocks is not None:
        local_first = [0]
        for lo, hi in blocks:
            local_first.append(local_first[-1] + hi - lo)
        log.set_blocks(local_first, [lo for lo, _ in blocks])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    join = None
    if world > 1 and args.join == "allgather":
        join = D.MatchExchange(ctx, dev)    # siesta_exchange_*: peer regions over NVLink, sizes in-band, decode on the GPU

    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev) if wl["bytes_per_event"] * E <= 2.6e8 else None

    def step_resident(keep=False):
        """One request; keep=True returns its result (DeviceMatches) beside the sizes for the caller to close."""
        if flush is not None:
            flush.add_(1)  # inputs smaller than L2: evict them between steps
        if join is not None:
            # scan of the shard + device-side all-gather: returns when this rank holds every rank's decoded columns
            dm, st = join.detect_allgather(log, nfa, flags)
            out = (st.local_traces, st.local_occurrences, st.local_events, dm.n_matches_emitted, dm.kernel_ms, st.k1_ms,
                   dm.n_traces, st.wait_ms + st.host_gap_ms + st.pull_ms, st.scan_ms, st.wait_ms, st.pull_ms, st.pulled_bytes, st.host_gap_ms,
                   st.n_blocks, st.eager, st.join_ms)
        else:
            dm = log.detect_device(nfa, flags=flags)
            out = (dm.n_traces, dm.n_occurrences, dm.n_events, dm.n_matches_emitted, dm.kernel_ms, dm.detect_ms, dm.n_traces, 0.0)
        if keep:
            return out, dm
        dm.close()
        return out

    sampler = ClockSampler(local_rank)
    sampler.start()          # before the warm-up: its own start-up must not land in the timed region
    for _ in range(args.warmup):
        r0 = step_resident()
    barrier()
    sampler.mark_begin()
    launches0 = api.kernel_launches()
    k_ms, d_ms, x_ms, lat_ms = [], [], [], []
    barrier()
    t0 = time.perf_counter()
    last = None     # --dump-outputs: the last timed step's result, written after the timed region
    for i in range(args.steps):
        ts0 = time.perf_counter()
        if args.dump_outputs and i == args.steps - 1:
            r, last = step_resident(keep=True)
        else:
            r = step_resident()
        lat_ms.append((time.perf_counter() - ts0) * 1e3)
        k_ms.append(r[4])
        d_ms.append(r[5])
        x_ms.append(r[7])
    barrier()
    wall = time.perf_counter() - t0
    if os.environ.get("SIESTA_BENCH_DEBUG"):
        print(f"[rank {rank}] step ms: {[round(x, 2) for x in lat_ms]} exchange ms: {[round(x, 2) for x in x_ms]}", file=sys.stderr, flush=True)
    launches = api.kernel_launches() - launches0
    clocks = sampler.stop()
    assert r[:4] == r0[:4], "result changed between steps"
    if last is not None:
        if rank == 0:     # at N > 1 every rank holds the same joined list of all ranks
            dump_outputs(last, local_rank, args.dump_outputs)
        last.close()

    t_step = torch.tensor([wall / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_step, op=dist.ReduceOp.MAX)
    sec_per_step = float(t_step.item())
    value = E_total / sec_per_step

    # ---- size-independent properties of the FULL result (outside the timed region; the oracle only sees the sample below)
    properties = None
    if world == 1 and not args.no_properties:
        properties = full_size_properties(log, nfa, flags, wl["states"], d_off, d_act, d_ts, local_rank)

    # ---- parity on the sample: the first SAMPLE_TRACES traces of the log live on rank 0; at N > 1 rank LAST decodes
    # them out of the joined list it received (the exchanged bytes are what is checked), at N = 1 rank 0 re-runs them
    ns = min(SAMPLE_TRACES, T if blocks is None else blocks[0][1] - blocks[0][0]) if rank == 0 else 0
    s_off = s_act = s_ts = None
    if rank == 0:
        e = int(d_off[ns].item())
        s_off, s_act, s_ts = d_off[:ns + 1].cpu().numpy(), d_act[:e].cpu().numpy(), d_ts[:e].cpu().numpy()
    parity = None
    if not args.no_cpu_baseline:
        if join is not None:
            # the LAST rank cuts the sample's traces out of the joined list it received over NVLink and hands them to
            # rank 0, which owns the sample's log and the oracle
            nsg = torch.tensor([ns], dtype=torch.int64, device=dev)
            dist.broadcast(nsg, 0)
            dm, _ = join.detect_allgather(log, nfa, flags)
            if rank == world - 1:
                D.send_columns(D.joined_prefix(dm.tensors(local_rank), int(nsg.item())), 0)
            if rank == 0:
                parity = ("pending", D.to_match_result(D.recv_columns(world - 1, dev)))
            dm.close()
        elif world == 1:
            plog = ctx.wrap_log(d_off[:ns + 1], d_act[:len(s_act)], d_ts[:len(s_ts)], wl["n_act"], max_trace_len=wl["max_len"])
            got = plog.detect(nfa, flags=flags)
            plog.close()
            parity = ("pending", got)

    # ---- e2e: the host-buffer C-ABI call (H2D of the events + verification + D2H of the occurrences) on a host slice
    e2e = None
    if not args.no_e2e:
        n_e = min(wl["e2e_traces"], T)
        e_e = int(d_off[n_e].item())
        h_off = torch.empty(n_e + 1, dtype=torch.int64).pin_memory()
        h_act = torch.empty(e_e, dtype=torch.int32).pin_memory()
        h_ts = torch.empty(e_e, dtype=torch.int64).pin_memory()
        h_off.copy_(d_off[:n_e + 1])
        h_act.copy_(d_act[:e_e])
        h_ts.copy_(d_ts[:e_e])
        torch.cuda.synchronize()
        np_off, np_act, np_ts = h_off.numpy(), h_act.numpy(), h_ts.numpy()
        # a query without a time constraint reads timestamps only for the events it reports, in place from the pinned host
        # column (siesta_evaluate_events): 4 B/event + 8 B per reported event / matching trace cross the link instead of 12 B/event
        ts_in_place = wl["bytes_per_event"] == 4 and not os.environ.get("SIESTA_NO_TS_ZERO_COPY")
        flags0 = flags

        def e2e_leg(col, act_bytes, call):
            flags = flags0 | args.e2e_extra_flags
            for _ in range(2):  # warm: stream-ordered pool, pinned result arena
                ctx.evaluate_events(np_off, col, np_ts, wl["n_act"], nfa, flags=flags, copy=False).close()
            barrier()
            t0 = time.perf_counter()
            for _ in range(max(1, args.e2e_steps)):
                res = ctx.evaluate_events(np_off, col, np_ts, wl["n_act"], nfa, flags=flags, copy=False)
                n_res = (res.n_traces, res.n_occurrences, res.n_events, int(res.trace_idx[-1]) if res.n_traces else -1)
                res.close()
            barrier()
            sec = (time.perf_counter() - t0) / max(1, args.e2e_steps)
            t_e2e = torch.tensor([sec], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
            sec = float(t_e2e.item())
            no_cols = bool(flags & abi.F_NO_EVENT_COLUMNS)
            h2d = 8 * (n_e + 1) + act_bytes * e_e + ((0 if no_cols else 8 * (n_res[2] + n_res[0])) if ts_in_place else 8 * e_e)
            d2h = 8 * n_res[0] + 8 * (n_res[0] + 1) + 8 * (n_res[1] + 1) + (4 if no_cols else 4 + 4 + 4 + 8) * n_res[2]
            return {"value": e_e * world / sec, "unit": "events/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": sec * 1e3, "bound": "pcie (host link: %.1f GB/s of payload%s)" % ((h2d + d2h) / sec / 1e9, "; the in-place timestamp reads are 8-byte transactions over the same link" if ts_in_place and not no_cols else ""),
                    "slice": f"first {n_e} traces ({e_e} events) of each rank's shard, pinned host memory",
                    "timestamps": "read in place from the pinned host column, reported events only" if ts_in_place else "copied to the device",
                    "call": call}

        e2e = e2e_leg(np_act, 4, "siesta_evaluate_events (pinned host CSR in, int32 activity column, chunked H2D overlapped with K1, host occurrences out)")
        if wl["n_act"] <= 256 and not args.e2e_int32:
            # the call runs at the speed of the host link, so the C-ABI also takes the activity column as one byte per event
            # (what the JNI serialiser writes for alphabets of at most 256 activities); the int32 call stays beside it
            h_act8 = torch.empty(e_e, dtype=torch.uint8).pin_memory()
            h_act8.copy_(d_act[:e_e].to(torch.uint8))
            torch.cuda.synchronize()
            wide = e2e
            e2e = e2e_leg(h_act8.numpy(), 1, "siesta_evaluate_events_act8 (pinned host CSR in, one byte per event for the activity column, "
                          "widened on the device, chunked H2D overlapped with K1, host occurrences out)")
            e2e["int32_column"] = {k: wide[k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "bound", "call")}
            del h_act8
        del h_off, h_act, h_ts

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        det_ms = float(np.mean(d_ms))
        # algorithmic bytes of one K1 launch on this rank (DESIGN.md §3): bytes_per_event x E (4: int32 activity;
        # 12 with the int64 timestamp when the query has a time constraint) + 8 B/trace offsets + the result
        # (8 B trace id + 8 + 8 B offsets per matching trace, 20 B per reported event)
        out_bytes = 8 * r[0] + 8 * (r[0] + 1) + 8 * (r[1] + 1) + 20 * r[2]
        alg_bytes = wl["bytes_per_event"] * E + 8 * T + out_bytes
        achieved = alg_bytes / (det_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic_bytes(args.workload, T)
        lat = np.array(lat_ms)
        line = {
            "metric": "events scanned/sec (/detection verification)", "value": value, "unit": "events/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": config_of(args, wl),
            "layout": {"traces_per_gpu": T, "events_per_gpu": E,
                       "parallelism": (f"traces sharded over {world} GPU(s) " +
                                       (f"block-cyclically ({args.blocks} blocks per rank of {blocks[0][1] - blocks[0][0]} traces)"
                                        if blocks is not None else "by contiguous range")) +
                                      ("; every rank ends the step with the decoded match list of all ranks in global trace order "
                                       "(pull + decode kernels over NVLink peer memory, sizes in-band" +
                                       (", block b pulled and decoded while block b + 1 is scanned)" if blocks is not None else ")")
                                       if join is not None else ""),
                       "l2": (f"inputs ({12 * E / 1e9:.2f} GB/GPU resident, {wl['bytes_per_event']} B/event read) "
                              + ("larger than L2; no flush needed" if flush is None else
                                 "SMALLER than L2: a 512 MB buffer is rewritten between steps"))},
            "roofline": {"bound": "hbm", "kernel": wl["kernel"],
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": det_ms, "all_kernels_ms": float(np.mean(k_ms))},
            "e2e": e2e,
            # one /detection request on the resident shard(s): wall time of the call on rank 0, result sizes back on the host
            "latency_ms": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                           "min": float(lat.min()), "max": float(lat.max()), "steps": [round(float(x), 3) for x in lat]},
            "p50_latency_ms": float(np.percentile(lat, 50)),
            "exchange": ({"ms": float(np.mean(x_ms)), "scan_and_place_ms": r[8], "wait_for_slowest_rank_ms": r[9],
                          "host_sizes_and_alloc_ms": r[12], "pull_and_decode_ms": r[10], "pulled_bytes_per_rank": r[11],
                          "nvlink_GBps_in": r[11] / max(r[15] if r[13] > 1 else r[10], 1e-9) / 1e6,
                          "blocks_per_rank": r[13], "eager_allocation": bool(r[14]), "join_stream_ms": r[15],
                          "what": "siesta_detect_allgather: compact blocks placed in peer-mapped regions, sizes in-band, pull + decode "
                                  "kernels on a second stream (block-cyclic shards: overlapped with the scan of the next block; "
                                  "pull_and_decode_ms is then what the join adds behind the last block), two host waits per request"}
                         if join is not None else None),
            "gpu_launches": launches,
            "clocks": clocks,
            "result": {"matching_traces_rank0": r[0], "occurrences_rank0": r[1], "events_rank0": r[2],
                       "matching_traces_all_ranks": r[6]},
        }
        if properties is not None:
            line["properties_full_size"] = properties
        if not args.no_cpu_baseline:
            import oracle
            t0 = time.perf_counter()
            want = oracle.detect(s_off, s_act, s_ts, nfa, flags=flags, n_threads=1)
            dt = time.perf_counter() - t0
            if isinstance(parity, tuple):
                ok, why = parity[1].same_as(want)
                parity = bool(ok)
            line["cpu_baseline"] = {"value": len(s_act) / dt, "unit": "events/s", "cores": 1, "kind": "port",
                                    "sample": f"first {ns} traces ({len(s_act)} events) of the same log, {dt:.1f} s",
                                    "parity_on_sample": parity}
        emit(line)
    log.close()
    if join is not None:
        join.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
