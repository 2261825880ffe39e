"""Multi-GPU plumbing: one process per GPU, traces sharded by contiguous trace range (SURVEY.md §8e).

The scan itself has no exchange step: every rank verifies / counts its own shard.  The results are joined afterwards:
- /detection: MatchExchange sets up the library's exchange (siesta_exchange_*, csrc/multi.cu) over torch.distributed;
  every request then all-gathers the per-rank match lists on the devices, over NVLink peer memory.
- /declare, /stats: a sum all-reduce of the packed int64 count array, on the devices (MatchExchange.allreduce_counts) or
  through torch.distributed (allreduce_counts, allreduce_pair_stats; these also work on CPU tensors with the gloo
  backend, tests/test_distributed_cpu.py).
"""
import numpy as np

import torch
import torch.distributed as dist

from . import _abi


def shard_bounds(trace_off, world):
    """Contiguous trace ranges balanced by event count: rank r owns traces [b[r], b[r+1])."""
    trace_off = np.asarray(trace_off, dtype=np.int64)
    T = len(trace_off) - 1
    E = int(trace_off[-1])
    targets = (np.arange(1, world, dtype=np.int64) * E) // world
    cuts = np.searchsorted(trace_off, targets, side="left").astype(np.int64)
    b = np.concatenate(([0], np.clip(cuts, 0, T), [T])).astype(np.int64)
    return np.maximum.accumulate(b)


def local_shard(trace_off, act, ts_ms, rank, world):
    """The CSR slice of rank `rank` (offsets rebased to 0) and the global index of its first trace."""
    b = shard_bounds(trace_off, world)
    lo, hi = int(b[rank]), int(b[rank + 1])
    e0, e1 = int(trace_off[lo]), int(trace_off[hi])
    return (np.asarray(trace_off[lo:hi + 1], dtype=np.int64) - e0, np.asarray(act[e0:e1]), np.asarray(ts_ms[e0:e1]), lo)


def allreduce_counts(packed, group=None):
    """Sum all-reduce of the packed int64 count array of siesta_declare_counts (in place)."""
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    return packed


def allreduce_pair_stats(packed, group=None):
    """Combine siesta_pair_stats_device results (int64[8 * n_pairs]: count, sum, min, max, four 32-bit limbs of the
    sum of squares) across ranks: SUM for count / sum / limbs, MIN / MAX for the extremes, then carry-normalise the
    limbs.  In place; returns the tensor."""
    v = packed.view(-1, 8)
    sums = v[:, [0, 1, 4, 5, 6, 7]].contiguous()
    mn = v[:, 2].contiguous()
    mx = v[:, 3].contiguous()
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(mn, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    limbs = sums[:, 2:6].clone()
    for k in range(3):
        carry = limbs[:, k] >> 32
        limbs[:, k] &= 0xFFFFFFFF
        limbs[:, k + 1] += carry
    v[:, 0], v[:, 1], v[:, 2], v[:, 3] = sums[:, 0], sums[:, 1], mn, mx
    v[:, 4:8] = limbs
    return packed


def pair_stats_records(packed):
    """packed int64[8 * n_pairs] (after allreduce_pair_stats) -> list of dicts like EventLog.pair_stats."""
    out = []
    for r in packed.view(-1, 8).cpu().tolist():
        cnt = r[0]
        sq = r[4] | (r[5] << 32) | (r[6] << 64) | (r[7] << 96)
        out.append({"count": cnt, "sum": r[1], "min": r[2] if cnt else 0, "max": r[3] if cnt else 0, "sum_squares": sq})
    return out


# ------------------------------------------------------------------------------------- exchange inside the library
class MatchExchange:
    """One process per GPU (torchrun): the library's own exchange (siesta_exchange_*, csrc/multi.cu) wired up over
    torch.distributed.  torch only carries the 64-byte IPC handles and the capacity agreement at set-up; every request
    afterwards runs inside libsiesta_gpu: the scan places its compact block in the rank's region, sizes travel in the
    block's header, one kernel pulls all peers' blocks over NVLink and decodes them to the joined columns."""

    def __init__(self, ctx, device, group=None):
        self.ctx, self.device, self.group = ctx, device, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.x = None
        self.capacity = 0

    def _ensure(self, need):
        """Collective: (re)create the exchanges when any rank needs a larger region."""
        t = torch.tensor([need], dtype=torch.int64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        need = int(t.item())
        if self.x is not None and need <= self.capacity:
            return
        from . import api
        if self.x is not None:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
            self.x.close()
        self.capacity = int(need * 1.25) + (1 << 20)
        self.x = api.Exchange(self.ctx, self.world, self.rank, self.capacity)
        mine = torch.frombuffer(bytearray(self.x.export()), dtype=torch.uint8).to(self.device)
        handles = torch.empty(self.world * mine.numel(), dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(handles, mine, group=self.group)
        handles = handles.cpu().view(self.world, -1)
        for p in range(self.world):
            if p != self.rank:
                self.x.import_peer(p, bytes(handles[p].numpy().tobytes()))
        dist.barrier(group=self.group)

    def detect_allgather(self, log, nfa, flags=0):
        """-> (api.DeviceMatches holding the match list of ALL ranks, ExchangeStats).  Collective."""
        from . import api
        key = (log.n_traces, log.n_events, bytes(nfa), flags)
        if getattr(self, "_sized_for", None) != key:
            self._ensure(api.exchange_required_bytes(log, nfa, flags))
            self._sized_for = key
        return self.x.detect_allgather(log, nfa, flags)

    def allreduce_counts(self, packed, op=_abi.REDUCE_SUM):
        if self.x is None or packed.numel() * 8 > self.capacity:
            self._ensure(packed.numel() * 8)
            self._sized_for = None
        return self.x.allreduce_i64(packed, op, torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if self.x is not None:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
            self.x.close()
            self.x = None


def joined_prefix(tensors, n_first_traces):
    """The part of a joined match list (dict of device tensors, DeviceMatches.tensors()) that belongs to global traces
    [0, n_first_traces): prefix slices, because the list is in trace order."""
    tr = tensors["trace_idx"]
    n = int(torch.searchsorted(tr, torch.tensor([n_first_traces], dtype=tr.dtype, device=tr.device)).item())
    n_occ = int(tensors["occ_off"][n].item()) if tensors["occ_off"].numel() else 0
    n_ev = int(tensors["ev_off"][n_occ].item()) if tensors["ev_off"].numel() else 0
    out = {"trace_idx": tr[:n], "occ_off": tensors["occ_off"][:n + 1], "ev_off": tensors["ev_off"][:n_occ + 1],
           "err_trace_idx": tensors["err_trace_idx"][tensors["err_trace_idx"] < n_first_traces]}
    for k in ("ev_pos", "ev_rank", "ev_act", "ev_ts_ms"):
        if k in tensors:
            out[k] = tensors[k][:n_ev]
    return out


_COLS = ("trace_idx", "occ_off", "ev_off", "err_trace_idx", "ev_pos", "ev_rank", "ev_act", "ev_ts_ms")
_DT = {"trace_idx": torch.int64, "occ_off": torch.int64, "ev_off": torch.int64, "ev_pos": torch.int32,
       "err_trace_idx": torch.int64, "ev_rank": torch.int32, "ev_act": torch.int32, "ev_ts_ms": torch.int64}


def send_columns(cols, dst, group=None):
    """Point-to-point transfer of a dict of 1-D tensors (sizes first); the receiver calls recv_columns."""
    dev = cols["trace_idx"].device
    sizes = torch.tensor([cols[k].numel() if k in cols else -1 for k in _COLS], dtype=torch.int64, device=dev)
    dist.send(sizes, dst, group=group)
    for k in _COLS:
        if k in cols and cols[k].numel():
            dist.send(cols[k].contiguous(), dst, group=group)


def recv_columns(src, device, group=None):
    sizes = torch.zeros(len(_COLS), dtype=torch.int64, device=device)
    dist.recv(sizes, src, group=group)
    out = {}
    for k, n in zip(_COLS, sizes.tolist()):
        if n < 0:
            continue
        t = torch.zeros(n, dtype=_DT[k], device=device)
        if n:
            dist.recv(t, src, group=group)
        out[k] = t
    return out


def to_match_result(g, n_matches_emitted=-1):
    """dict of tensors -> host MatchResult (for comparison with the oracle)."""
    r = _abi.MatchResult()
    h = {k: v.cpu().numpy() for k, v in g.items()}
    r.trace_idx, r.occ_off, r.ev_off, r.err_trace_idx = h["trace_idx"], h["occ_off"], h["ev_off"], h["err_trace_idx"]
    r.ev_pos = h.get("ev_pos")
    r.ev_rank, r.ev_act, r.ev_ts_ms = h.get("ev_rank"), h.get("ev_act"), h.get("ev_ts_ms")
    r.n_traces, r.n_occurrences, r.n_events = len(r.trace_idx), len(r.ev_off) - 1, int(r.ev_off[-1])
    r.n_ref_errors, r.n_matches_emitted, r.kernel_ms, r.detect_ms = len(r.err_trace_idx), n_matches_emitted, 0.0, 0.0
    r.unsupported_trace_idx = h.get("unsupported_trace_idx", np.zeros(0, dtype=np.int64))
    r.n_unsupported = len(r.unsupported_trace_idx)
    return r

