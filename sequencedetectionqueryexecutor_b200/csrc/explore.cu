// explore.cu — /explore in accurate mode (row X): for every candidate continuation, the exact number of occurrences
// of pattern + candidate and the summed duration of those occurrences.
//
// Replaces QueryPlanExplorationAccurate.patternDetection (J/model/Queries/QueryPlans/Exploration/
// QueryPlanExplorationAccurate.java:82-102): SimplePattern + [next] -> SaseConnector.evaluate(..., false) ->
// clearOccurrences(true) per trace -> completions = number of occurrences, average duration =
// sum(Occurrence.getDuration) / completions with getDuration = (last.ms - first.ms) / 1000.0 (J/model/Occurrence.java:
// 55-61).  The reference runs one full detection per candidate.  Here ONE pass over the log serves all candidates:
// the extended pattern p1 .. pm x has only normal states and no predicates (class NK), so the run started at an event of
// p1 takes greedily the first later p2, p3 ... pm - the same for every candidate - and then the first later x.
//   explore_prefix_kernel  one warp per trace, lanes = events (coalesced 4 B/event): position masks of p1 .. pm by ballot,
//                          the greedy prefix walk of every start -> a record (start slots, prefix-end slots) for the few
//                          traces that hold the prefix at all
//   explore_tail_kernel    one lane per (recorded trace, candidate): position mask of the candidate, completion of every
//                          start, Occurrences.clearOccurrences(true) (first in emission order + the later ones that overlap
//                          nothing chosen, J/model/Occurrences.java:58-89, Occurrence.overlaps :36-49) and the durations
// Emission order is (completion, start); prefix ends and therefore completions never decrease with the start, so it is
// the order of the starts.  Traces that do not fit the fast path (more than 64 events or more than 16 starts) are put on
// an overflow list and evaluated by the general kernels (one detection per candidate over just those traces).
// The library returns exact integers (completions, summed milliseconds); the double division stays with the caller.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

namespace siesta {

__global__ void __launch_bounds__(256) occurrence_duration_kernel(const int64_t* ev_off, const int64_t* ev_ts, int64_t n_occ,
                                                                  unsigned long long* sum_ms) {
    long long acc = 0;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_occ; o += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = ev_off[o], b = ev_off[o + 1];
        if (b > a) acc += ev_ts[b - 1] - ev_ts[a];
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const int lo = __shfl_xor_sync(0xffffffffu, (int)(acc & 0xffffffffll), d);
        const int hi = __shfl_xor_sync(0xffffffffu, (int)(acc >> 32), d);
        acc += ((long long)hi << 32) | (unsigned int)lo;
    }
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(sum_ms, (unsigned long long)acc);
}


constexpr int EX_STARTS = 16;  // starts of a trace the record holds

struct ExploreRecord {   // 48 bytes
    int64_t trace;
    uint8_t n, first_pat, pad[6];
    uint8_t s[EX_STARTS], e[EX_STARTS];
};

struct ExploreParams {
    const int64_t* trace_off;
    const int32_t* act;
    const int64_t* ts_ms;
    int64_t n_traces;
    int32_t m;                       // pattern length
    int32_t pat[SIESTA_MAX_STATES];
    ExploreRecord* rec;
    int64_t* ovf;                    // traces for the general kernels
    unsigned long long* counters;    // 0 records, 1 overflow
    // tail
    const int32_t* cand;
    int32_t n_cand;
    int32_t evt_pos;
    unsigned long long* comp;
    unsigned long long* sum_ms;
};

__device__ __forceinline__ long long ex_shfl64(long long v, int src) {
    int lo = __shfl_sync(0xffffffffu, (int)(v & 0xffffffffll), src);
    int hi = __shfl_sync(0xffffffffu, (int)(v >> 32), src);
    return ((long long)hi << 32) | (unsigned int)lo;
}

constexpr int EX_BATCH = 4;  // traces a warp has in flight (their loads are issued before the first is used)

__global__ void __launch_bounds__(256) explore_prefix_kernel(const __grid_constant__ ExploreParams P) {
    const int lane = threadIdx.x & 31;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long tb = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * EX_BATCH; tb < P.n_traces;
         tb += warps_total * EX_BATCH) {
        // offsets of the batch: lane k holds trace_off[tb + k], k = 0 .. EX_BATCH
        long long myoff = 0;
        if (lane <= EX_BATCH && tb + lane <= P.n_traces) myoff = P.trace_off[tb + lane];
        long long lo[EX_BATCH], len[EX_BATCH];
        int a0[EX_BATCH], a1[EX_BATCH];
#pragma unroll
        for (int u = 0; u < EX_BATCH; ++u) {
            lo[u] = ex_shfl64(myoff, u);
            const long long hi = ex_shfl64(myoff, u + 1);
            len[u] = tb + u < P.n_traces ? hi - lo[u] : 0;
            a0[u] = (len[u] <= 64 && lane < len[u]) ? __ldg(P.act + lo[u] + lane) : -1;
            a1[u] = (len[u] <= 64 && 32 + lane < len[u]) ? __ldg(P.act + lo[u] + 32 + lane) : -1;
        }
#pragma unroll
        for (int u = 0; u < EX_BATCH; ++u) {
            const long long t = tb + u;
            if (len[u] <= 0) continue;
            if (len[u] > 64) {
                if (lane == 0) P.ovf[atomicAdd(P.counters + 1, 1ull)] = t;
                continue;
            }
            unsigned long long T[SIESTA_MAX_STATES];
            bool all = true;
#pragma unroll
            for (int k = 0; k < SIESTA_MAX_STATES; ++k) {
                T[k] = 0;
                if (k < P.m) {
                    const int x = P.pat[k];
                    T[k] = (unsigned long long)__ballot_sync(0xffffffffu, a0[u] == x) |
                           ((unsigned long long)__ballot_sync(0xffffffffu, a1[u] == x) << 32);
                    all = all && T[k] != 0;
                }
            }
            if (!all) continue;  // uniform: the prefix's activities do not all occur
            // greedy prefix walk of every start (uniform: every lane computes the same; lane 0 writes)
            unsigned long long uni = 0;
#pragma unroll
            for (int k = 0; k < SIESTA_MAX_STATES; ++k) uni |= T[k];
            ExploreRecord r;
            r.trace = t;
            r.n = 0;
            r.first_pat = (uint8_t)(__ffsll((long long)uni) - 1);
            bool too_many = false;
            for (unsigned long long st = T[0]; st; st &= st - 1) {
                const unsigned long long sb = st & (0ull - st);
                unsigned long long pb = sb;
                bool ok = true;
#pragma unroll
                for (int k = 1; k < SIESTA_MAX_STATES; ++k) {
                    if (k < P.m && ok) {
                        const unsigned long long c = T[k] & ~(pb | (pb - 1));
                        if (!c) ok = false;
                        else pb = c & (0ull - c);
                    }
                }
                if (!ok) break;  // prefix ends never decrease with the start: a later start fails as well
                if (r.n == EX_STARTS) { too_many = true; break; }
                r.s[r.n] = (uint8_t)(__ffsll((long long)sb) - 1);
                r.e[r.n] = (uint8_t)(__ffsll((long long)pb) - 1);
                ++r.n;
            }
            if (too_many) {
                if (lane == 0) P.ovf[atomicAdd(P.counters + 1, 1ull)] = t;
            } else if (r.n && lane == 0) {
                P.rec[atomicAdd(P.counters + 0, 1ull)] = r;
            }
        }
    }
}

// lanes of a warp = 32 candidates of ONE recorded trace (the trace's events are uniform, broadcast loads)
__global__ void __launch_bounds__(256) explore_tail_kernel(const __grid_constant__ ExploreParams P, long long n_rec) {
    const int lane = threadIdx.x & 31;
    const int groups = (P.n_cand + 31) / 32;
    const long long items = n_rec * groups;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long it = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); it < items; it += warps_total) {
        const ExploreRecord& R = P.rec[it / groups];
        const int ci = (int)(it % groups) * 32 + lane;
        const int x = ci < P.n_cand ? P.cand[ci] : -2;
        const long long lo = P.trace_off[R.trace];
        const int len = (int)(P.trace_off[R.trace + 1] - lo);
        unsigned long long Mx = 0;
        for (int i = 0; i < len; ++i)
            if (__ldg(P.act + lo + i) == x) Mx |= 1ull << i;
        if (!Mx || x < 0) continue;
        const long long* ts = reinterpret_cast<const long long*>(P.ts_ms) + lo;
        // first event of the filtered list (pattern activities + candidate): Utils.java:51-53
        const int first_x = __ffsll((long long)Mx) - 1;
        const long long t0 = __ldg(ts + (first_x < (int)R.first_pat ? first_x : (int)R.first_pat));
        // attribute Occurrence.overlaps compares: in-trace position (EventPos route) or relative seconds (EventTs route)
        auto attr = [&](int slot) -> long long {
            if (P.evt_pos) return slot;
            return (long long)(int)((__ldg(ts + slot) - t0) / 1000);   // EventTs.java:54: truncating division
        };
        long long sel_s[EX_STARTS], sel_c[EX_STARTS];  // attribute of the first / last event of the chosen occurrences
        int nsel = 0;
        long long dur = 0;
        for (int i = 0; i < (int)R.n; ++i) {
            const unsigned long long c = Mx & (~1ull << R.e[i]);
            if (!c) break;  // completions never decrease with the start either
            const int cs = __ffsll((long long)c) - 1;
            const long long as = attr(R.s[i]), ac = attr(cs);
            bool ov = false;
            for (int o = 0; o < nsel && !ov; ++o) ov = !(ac < sel_s[o] || as > sel_c[o]);
            if (ov) continue;
            sel_s[nsel] = as;
            sel_c[nsel] = ac;
            ++nsel;
            // Occurrence.getDuration on SaseEvent.getEventBoth's timestamps (timestamp * 1000 + minTs on the EventTs route)
            dur += P.evt_pos ? (__ldg(ts + cs) - __ldg(ts + R.s[i])) : (ac - as) * 1000;
        }
        if (nsel) {
            atomicAdd(P.comp + ci, (unsigned long long)nsel);
            atomicAdd(P.sum_ms + ci, (unsigned long long)dur);
        }
    }
}

}  // namespace siesta

using namespace siesta;

extern "C" int siesta_explore_accurate(siesta_log* log, const int32_t* pattern_activities, int32_t n_pattern,
                                       const int32_t* candidates, int32_t n_candidates, uint32_t flags,
                                       int64_t* completions, int64_t* sum_duration_ms, double* kernel_ms) {
    Log* L = reinterpret_cast<Log*>(log);
    if (!L || !pattern_activities || n_pattern < 1 || n_pattern + 1 > SIESTA_MAX_STATES || (n_candidates && !candidates) ||
        n_candidates < 0 || !completions || !sum_duration_ms) {
        set_error("siesta_explore_accurate: bad argument (pattern of 1.." + std::to_string(SIESTA_MAX_STATES - 1) + " events)");
        return SIESTA_E_INVALID;
    }
    if (flags & ~(uint32_t)SIESTA_F_EVT_POS) {
        set_error("siesta_explore_accurate: only SIESTA_F_EVT_POS may be set (returnAll is implied)");
        return SIESTA_E_INVALID;
    }
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    cudaStream_t stream = L->ctx->stream;
    const int64_t T = L->n_traces;
    const size_t nc = (size_t)(n_candidates ? n_candidates : 1);
    // one allocation: comp[nc] sum[nc] counters[2] cand[nc] | overflow list [T] | records [T]
    unsigned long long* d_acc = nullptr;
    const size_t acc_words = 2 * nc + 2;
    const size_t cand_off = (acc_words * 8 + 255) & ~(size_t)255;
    const size_t ovf_off = (cand_off + nc * 4 + 255) & ~(size_t)255;
    const size_t rec_off = (ovf_off + (size_t)std::max<int64_t>(T, 1) * 8 + 255) & ~(size_t)255;
    const size_t total = rec_off + (size_t)std::max<int64_t>(T, 1) * sizeof(ExploreRecord);
    cudaError_t ce = cudaMallocAsync((void**)&d_acc, total, stream);
    if (ce != cudaSuccess) {
        set_error(std::string("siesta_explore_accurate: cudaMalloc: ") + cudaGetErrorString(ce));
        return SIESTA_E_NOMEM;
    }
    char* base = reinterpret_cast<char*>(d_acc);
    SIESTA_CUDA_OK(cudaMemsetAsync(d_acc, 0, acc_words * 8, stream));
    if (n_candidates) SIESTA_CUDA_OK(cudaMemcpyAsync(base + cand_off, candidates, (size_t)n_candidates * 4, cudaMemcpyHostToDevice, stream));
    cudaEvent_t e0, e1;
    SIESTA_CUDA_OK(cudaEventCreate(&e0));
    SIESTA_CUDA_OK(cudaEventCreate(&e1));
    SIESTA_CUDA_OK(cudaEventRecord(e0, stream));
    ExploreParams P;
    std::memset(&P, 0, sizeof(P));
    P.trace_off = L->d_trace_off;
    P.act = L->d_act;
    P.ts_ms = L->d_ts_ms;
    P.n_traces = T;
    P.m = n_pattern;
    for (int k = 0; k < n_pattern; ++k) P.pat[k] = pattern_activities[k];
    P.rec = reinterpret_cast<ExploreRecord*>(base + rec_off);
    P.ovf = reinterpret_cast<int64_t*>(base + ovf_off);
    P.counters = d_acc + 2 * nc;
    P.cand = reinterpret_cast<const int32_t*>(base + cand_off);
    P.n_cand = n_candidates;
    P.evt_pos = (flags & SIESTA_F_EVT_POS) ? 1 : 0;
    P.comp = d_acc;
    P.sum_ms = d_acc + nc;
    unsigned long long h_cnt[2] = {0, 0};
    if (T > 0 && n_candidates > 0) {
        const int grid = (int)std::min<int64_t>((T + 8 * EX_BATCH - 1) / (8 * EX_BATCH), (int64_t)L->ctx->sm_count * 8);
        explore_prefix_kernel<<<grid, 256, 0, stream>>>(P);
        SIESTA_LAUNCHED();
        SIESTA_CUDA_OK(cudaGetLastError());
        SIESTA_CUDA_OK(cudaMemcpyAsync(h_cnt, P.counters, 16, cudaMemcpyDeviceToHost, stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
        if (h_cnt[0] > 0) {
            const long long items = (long long)h_cnt[0] * ((n_candidates + 31) / 32);
            const int grid2 = (int)std::min<long long>((items + 7) / 8, (long long)L->ctx->sm_count * 8);
            explore_tail_kernel<<<grid2, 256, 0, stream>>>(P, (long long)h_cnt[0]);
            SIESTA_LAUNCHED();
            SIESTA_CUDA_OK(cudaGetLastError());
        }
    }
    SIESTA_CUDA_OK(cudaEventRecord(e1, stream));
    std::vector<unsigned long long> h_acc(2 * nc);
    SIESTA_CUDA_OK(cudaMemcpyAsync(h_acc.data(), d_acc, 2 * nc * 8, cudaMemcpyDeviceToHost, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    float fms = 0.f;
    cudaEventElapsedTime(&fms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    double ms = fms;
    for (int c = 0; c < n_candidates; ++c) {
        completions[c] = (int64_t)h_acc[c];
        sum_duration_ms[c] = (int64_t)h_acc[nc + c];
    }
    int rc = SIESTA_OK;
    // traces outside the fast path: one general detection per candidate over just those traces
    if (h_cnt[1] > 0) {
        const int64_t n_ovf = (int64_t)h_cnt[1];
        std::vector<int64_t> h_ovf((size_t)n_ovf);   // the general kernels want ascending candidates
        SIESTA_CUDA_OK(cudaMemcpyAsync(h_ovf.data(), P.ovf, (size_t)n_ovf * 8, cudaMemcpyDeviceToHost, stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
        std::sort(h_ovf.begin(), h_ovf.end());
        SIESTA_CUDA_OK(cudaMemcpyAsync(P.ovf, h_ovf.data(), (size_t)n_ovf * 8, cudaMemcpyHostToDevice, stream));
        unsigned long long* d_one = d_acc + 2 * nc;  // the counters are free again
        for (int c = 0; c < n_candidates && rc == SIESTA_OK; ++c) {
            siesta_nfa nfa;  // SimplePattern.getNfa: all states "normal" (J/model/Patterns/SimplePattern.java:96-104)
            std::memset(&nfa, 0, sizeof(nfa));
            nfa.n_states = n_pattern + 1;
            for (int st = 0; st <= n_pattern; ++st) {
                nfa.states[st].kind = SIESTA_STATE_NORMAL;
                nfa.states[st].n_types = 1;
                nfa.states[st].types[0] = st < n_pattern ? pattern_activities[st] : candidates[c];
            }
            siesta_dev_matches dm;
            rc = detect_device_impl(L, &nfa, P.ovf, n_ovf, flags | SIESTA_F_RETURN_ALL, stream, RebaseOffsets{0, 0, 0}, &dm);
            if (rc) break;
            ms += dm.kernel_ms;
            if (dm.n_ref_errors) {
                set_error("siesta_explore_accurate: the reference engine throws on this pattern");
                rc = SIESTA_E_REFERENCE_THROWS;
            } else if (dm.n_unsupported) {   // an aggregate over all traces cannot leave some out
                set_error("siesta_explore_accurate: " + std::to_string(dm.n_unsupported) + " trace(s) exceed the engine limits (siesta_detect lists them)");
                rc = SIESTA_E_UNSUPPORTED;
            } else if (dm.n_occurrences > 0) {
                completions[c] += dm.n_occurrences;
                SIESTA_CUDA_OK(cudaMemsetAsync(d_one, 0, 8, stream));
                const int grid = (int)std::min<int64_t>((dm.n_occurrences + 255) / 256, (int64_t)L->ctx->sm_count * 8);
                occurrence_duration_kernel<<<grid, 256, 0, stream>>>(dm.d_ev_off, dm.d_ev_ts_ms, dm.n_occurrences, d_one);
                SIESTA_LAUNCHED();
                unsigned long long h_one = 0;
                SIESTA_CUDA_OK(cudaMemcpyAsync(&h_one, d_one, 8, cudaMemcpyDeviceToHost, stream));
                SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
                sum_duration_ms[c] += (int64_t)h_one;
            }
            siesta_dev_matches_free(&dm);
        }
    }
    cudaFreeAsync(d_acc, stream);
    if (kernel_ms) *kernel_ms = ms;
    return rc;
}
