// append.cu — growing a resident log on the device: siesta_log_append and siesta_log_read (siesta_multi_log_append,
// in multi.cu, runs siesta_log_append on every shard).
//
// A batch that touches k traces (listed trace i gets batch events [batch_off[i], batch_off[i + 1]) after its old
// events) turns the old columns into 2k + 1 pieces of the new ones:
//   old run i (i = 0..k)   old events [P[i - 1], P[i]) (P[-1] = 0), moved right by batch_off[i]
//   batch i   (i = 0..k-1) batch events [batch_off[i], batch_off[i + 1]), placed at P[i] + batch_off[i]
// where P[i] = old_off[min(trace_idx[i] + 1, T)] is the old event before which batch i goes in (P[k] = E).  In the new
// columns old run i ends at D[i] = P[i] + batch_off[i] and batch i at end[i] = P[i] + batch_off[i + 1]; both ascend, so
// a block finds the piece an output position lies in by one binary search over end[].  The rebuild is a segmented copy:
// bound by HBM bandwidth, no scan beyond the caller's batch offsets.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

namespace siesta {

constexpr int64_t AP_TILE = 8192;   // output events per block of the copy kernel

// One thread per trace of the new log (and one for the closing offset): new_off[t] = old_off[min(t, T)] + batch_off[j]
// with j = listed traces below t (binary search over trace_idx, which stays in L2).  Also writes P[] for the listed
// traces and reduces the longest new trace.
__global__ void __launch_bounds__(AP_T) ap_offsets_kernel(const int64_t* __restrict__ old_off, int64_t T, int64_t T2,
                                                         const int64_t* __restrict__ tidx, const int64_t* __restrict__ boff,
                                                         int64_t k, int64_t* __restrict__ new_off, int64_t* __restrict__ P,
                                                         unsigned long long* max_len) {
    const int64_t t = (int64_t)blockIdx.x * AP_T + threadIdx.x;
    unsigned long long len = 0;
    if (t <= T2) {
        int64_t lo = 0, hi = k;   // j = first listed index with tidx[j] >= t
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (tidx[mid] < t) lo = mid + 1; else hi = mid;
        }
        const int64_t o = old_off[t < T ? t : T];
        new_off[t] = o + boff[lo];
        if (t < T2) {
            const int64_t o1 = t < T ? old_off[t + 1] : o;
            const bool listed = lo < k && tidx[lo] == t;
            len = (unsigned long long)(o1 - o + (listed ? boff[lo + 1] - boff[lo] : 0));
            if (listed) P[lo] = o1;
        } else {
            P[k] = o;   // t == T2: o = E
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, d));
    if ((threadIdx.x & 31) == 0 && len) atomicMax(max_len, len);
}

// Grid over the output columns, AP_TILE events per block.  The block finds the first piece that reaches into its tile
// by binary search, then walks the pieces of the tile.  Batch segments with no old event between them (new traces,
// consecutive listed traces whose old runs are empty) are one contiguous copy.
__global__ void __launch_bounds__(AP_T) ap_copy_kernel(const int32_t* __restrict__ old_act, const int64_t* __restrict__ old_ts,
                                                      const int32_t* __restrict__ b_act, const int64_t* __restrict__ b_ts,
                                                      const int64_t* __restrict__ P, const int64_t* __restrict__ boff, int64_t k,
                                                      int64_t E2, int32_t* __restrict__ o_act, int64_t* __restrict__ o_ts) {
    const int64_t o0 = (int64_t)blockIdx.x * AP_TILE;
    const int64_t o1 = o0 + AP_TILE < E2 ? o0 + AP_TILE : E2;
    auto end_of = [&](int64_t i) { return i < k ? P[i] + boff[i + 1] : E2; };
    int64_t lo = 0, hi = k;   // first piece pair i whose batch segment ends after o0
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (end_of(mid) <= o0) lo = mid + 1; else hi = mid;
    }
    int64_t i = lo, o = o0;
    while (o < o1) {
        const int64_t p = P[i], d = p + boff[i];   // old run i = output [.., d)
        if (o < d) {
            const int64_t n = (d < o1 ? d : o1) - o, s = o - boff[i];
            ap_copy(o_act + o, old_act + s, n);
            ap_copy(o_ts + o, old_ts + s, n);
            o += n;
        }
        if (o >= o1 || i >= k) break;
        int64_t j = i + 1;   // batch segments i .. j-1 share P (no old event between them): one source run
        {
            int64_t a = i + 1, b = k;
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                if (P[mid] == p) a = mid + 1; else b = mid;
            }
            j = a;
        }
        const int64_t e = p + boff[j];   // end of batch segment j - 1
        const int64_t n = (e < o1 ? e : o1) - o, s = o - p;
        if (n > 0) {
            ap_copy(o_act + o, b_act + s, n);
            ap_copy(o_ts + o, b_ts + s, n);
            o += n;
        }
        i = j;
    }
}

static size_t ap_align(size_t v) { return (v + 255) & ~(size_t)255; }

bool append_check_batch(const char* fn, int64_t T, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                        const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces) {
    if (!batch_off || n_listed < 0 || (n_listed > 0 && !trace_idx)) {
        set_error(std::string(fn) + ": null argument");
        return false;
    }
    if (n_new_traces < 0) {
        set_error(std::string(fn) + ": n_new_traces must be >= 0");
        return false;
    }
    if (batch_off[0] != 0) {
        set_error(std::string(fn) + ": batch_off[0] must be 0");
        return false;
    }
    for (int64_t i = 0; i < n_listed; ++i) {
        if (batch_off[i + 1] < batch_off[i]) {
            set_error(std::string(fn) + ": batch_off must be non-decreasing");
            return false;
        }
        if (trace_idx[i] < 0 || trace_idx[i] >= T + n_new_traces || (i > 0 && trace_idx[i] <= trace_idx[i - 1])) {
            set_error(std::string(fn) + ": trace_idx must ascend strictly inside [0, n_traces + n_new_traces)");
            return false;
        }
    }
    if (batch_off[n_listed] > 0 && (!act || !ts_ms)) {
        set_error(std::string(fn) + ": null event column");
        return false;
    }
    return true;
}

}  // namespace siesta

using namespace siesta;

extern "C" int siesta_log_append(siesta_log* log, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                                 const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces, int32_t n_activities,
                                 siesta_log** out, double* kernel_ms) {
    Log* S = reinterpret_cast<Log*>(log);
    if (!S || !out) {
        set_error("siesta_log_append: null argument");
        return SIESTA_E_INVALID;
    }
    if (S->d_src_event || S->n_blocks > 0) {
        set_error("siesta_log_append: derived (filter / group) and block-cyclic logs cannot grow");
        return SIESTA_E_INVALID;
    }
    if (n_activities < S->n_activities) {
        set_error("siesta_log_append: n_activities is smaller than the log's (the dictionary only grows)");
        return SIESTA_E_INVALID;
    }
    const int64_t T = S->n_traces, E = S->n_events;
    if (!append_check_batch("siesta_log_append", T, trace_idx, batch_off, n_listed, act, ts_ms, n_new_traces)) return SIESTA_E_INVALID;
    const int64_t k = n_listed, NB = batch_off[k], T2 = T + n_new_traces, E2 = E + NB;
    Ctx* c = S->ctx;
    SIESTA_CUDA_OK(cudaSetDevice(c->device));
    cudaStream_t stream = c->stream;

    // the new log's columns (tail padding as siesta_log_filter_time: whole 32-byte sectors may be read past the end)
    int64_t* d_off = nullptr;
    int32_t* d_act = nullptr;
    int64_t* d_ts = nullptr;
    const size_t ne = (size_t)(E2 ? E2 : 1);
    cudaError_t e;
    if ((e = cudaMalloc((void**)&d_off, (size_t)(T2 + 1) * 8 + 32)) != cudaSuccess || (e = cudaMalloc((void**)&d_act, ne * 4 + 32)) != cudaSuccess ||
        (e = cudaMalloc((void**)&d_ts, ne * 8 + 32)) != cudaSuccess) {
        cudaGetLastError();
        set_error(std::string("siesta_log_append: cudaMalloc: ") + cudaGetErrorString(e));
        cudaFree(d_off); cudaFree(d_act); cudaFree(d_ts);
        return SIESTA_E_NOMEM;
    }
    // staging: trace_idx, batch_off, P, act, ts, max length
    const size_t s_tidx = 0, s_boff = s_tidx + ap_align((size_t)std::max<int64_t>(k, 1) * 8), s_p = s_boff + ap_align((size_t)(k + 1) * 8),
                 s_act = s_p + ap_align((size_t)(k + 1) * 8), s_ts = s_act + ap_align((size_t)std::max<int64_t>(NB, 1) * 4 + 32),
                 s_max = s_ts + ap_align((size_t)std::max<int64_t>(NB, 1) * 8 + 32), s_all = s_max + 256;
    char* stage = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    auto fail = [&](int rc, const std::string& why) {
        cudaGetLastError();
        set_error("siesta_log_append: " + why);
        cudaStreamSynchronize(stream);
        if (stage) cudaFreeAsync(stage, stream);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        cudaFree(d_off); cudaFree(d_act); cudaFree(d_ts);
        return rc;
    };
    if ((e = cudaMallocAsync((void**)&stage, s_all, stream)) != cudaSuccess) {
        stage = nullptr;
        return fail(SIESTA_E_NOMEM, std::string("staging cudaMallocAsync: ") + cudaGetErrorString(e));
    }
    int64_t* d_tidx = reinterpret_cast<int64_t*>(stage + s_tidx);
    int64_t* d_boff = reinterpret_cast<int64_t*>(stage + s_boff);
    int64_t* d_P = reinterpret_cast<int64_t*>(stage + s_p);
    int32_t* d_bact = reinterpret_cast<int32_t*>(stage + s_act);
    int64_t* d_bts = reinterpret_cast<int64_t*>(stage + s_ts);
    unsigned long long* d_max = reinterpret_cast<unsigned long long*>(stage + s_max);
    e = cudaMemsetAsync(d_max, 0, 8, stream);
    if (e == cudaSuccess && k) e = cudaMemcpyAsync(d_tidx, trace_idx, (size_t)k * 8, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_boff, batch_off, (size_t)(k + 1) * 8, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess && NB) e = cudaMemcpyAsync(d_bact, act, (size_t)NB * 4, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess && NB) e = cudaMemcpyAsync(d_bts, ts_ms, (size_t)NB * 8, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaEventCreate(&ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&ev1);
    if (e == cudaSuccess) e = cudaEventRecord(ev0, stream);
    if (e != cudaSuccess) return fail(SIESTA_E_CUDA, std::string("batch staging: ") + cudaGetErrorString(e));

    ap_offsets_kernel<<<(unsigned)((T2 + 1 + AP_T - 1) / AP_T), AP_T, 0, stream>>>(S->d_trace_off, T, T2, d_tidx, d_boff, k, d_off, d_P, d_max);
    SIESTA_LAUNCHED();
    if (E2 > 0) {
        ap_copy_kernel<<<(unsigned)((E2 + AP_TILE - 1) / AP_TILE), AP_T, 0, stream>>>(S->d_act, S->d_ts_ms, d_bact, d_bts, d_P, d_boff, k, E2,
                                                                                     d_act, d_ts);
        SIESTA_LAUNCHED();
    }
    unsigned long long h_max = 0;
    if ((e = cudaGetLastError()) == cudaSuccess) e = cudaEventRecord(ev1, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_max, d_max, 8, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ev0, ev1);
    if (e != cudaSuccess) return fail(SIESTA_E_CUDA, std::string("rebuild: ") + cudaGetErrorString(e));

    // one range check of the batch ids against the new dictionary size (the old events were checked when they arrived)
    Log batch;
    batch.ctx = c;
    batch.d_act = d_bact;
    batch.n_activities = n_activities;
    batch.act_valid = true;
    if (validate_act_range(&batch, 0, NB, stream) != SIESTA_OK) return fail(SIESTA_E_CUDA, siesta_last_error());
    cudaFreeAsync(stage, stream);
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);

    Log* L = new Log();
    L->ctx = c;
    L->d_trace_off = d_off;
    L->d_act = d_act;
    L->d_ts_ms = d_ts;
    L->n_traces = T2;
    L->n_events = E2;
    L->n_activities = n_activities;
    L->max_trace_len = (int32_t)(h_max > 0x7fffffffull ? 0x7fffffffull : h_max);
    L->true_max_len = (int64_t)h_max;
    L->owns = true;
    L->first_trace = S->first_trace;
    L->act_valid = S->act_valid && batch.act_valid;
    if (kernel_ms) *kernel_ms = ms;
    *out = reinterpret_cast<siesta_log*>(L);
    return SIESTA_OK;
}

extern "C" int siesta_log_read(siesta_log* log, int64_t t0, int64_t t1, int64_t* trace_off, int32_t* act, int64_t* ts_ms) {
    Log* L = reinterpret_cast<Log*>(log);
    if (!L || !trace_off || (!act) != (!ts_ms)) {
        set_error("siesta_log_read: null argument (act and ts_ms are both given or both NULL)");
        return SIESTA_E_INVALID;
    }
    if (t0 < 0 || t1 < t0 || t1 > L->n_traces) {
        set_error("siesta_log_read: need 0 <= t0 <= t1 <= n_traces");
        return SIESTA_E_INVALID;
    }
    Ctx* c = L->ctx;
    SIESTA_CUDA_OK(cudaSetDevice(c->device));
    SIESTA_CUDA_OK(cudaMemcpyAsync(trace_off, L->d_trace_off + t0, (size_t)(t1 - t0 + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(c->stream));
    const int64_t e0 = trace_off[0], n = trace_off[t1 - t0] - e0;
    if (act && n > 0) {
        SIESTA_CUDA_OK(cudaMemcpyAsync(act, L->d_act + e0, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
        SIESTA_CUDA_OK(cudaMemcpyAsync(ts_ms, L->d_ts_ms + e0, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(c->stream));
    }
    return SIESTA_OK;
}
