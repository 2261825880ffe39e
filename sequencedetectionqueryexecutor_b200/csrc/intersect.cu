// intersect.cu — kernel K2: the pair index over a resident CSR log and the sorted trace-id intersection.
//
// Replaces SparkDatabaseRepository.getCommonIds (J/storage/repositories/SparkDatabaseRepository.java:160-178):
// "the traces that contain ALL true pairs" = intersection of the per-pair posting lists, each an ascending,
// duplicate-free list of dense trace indices.  Posting lists either come from the caller (index.parquet, loaded
// with siesta_index_load) or are derived on the GPU from the CSR log under the SeqTable view (siesta_index_build):
// a trace is listed under (A,B) iff it holds an A before a B (A == B: at least two occurrences).
//
// Kernels
//   pair_flags_kernel   one warp per trace: first / last position and count of the (<= 32) activities the requested
//                       pairs mention, then one lane per pair writes flag[pair][trace]
//   list_hits_kernel    one thread per element of every list: hit[trace] += 1 (byte counters, word atomics); a trace is in
//                       the intersection of n duplicate-free lists iff its counter reaches n: every list is read
//                       exactly once, coalesced (8 B x sum |list_i|), no search
//   compaction          block counts -> one-block scan -> ordered write (ascending output, deterministic)
//   index_dup_kernel    one thread per element of the delta lists of an index refresh / append: rank in its old list (one
//                       binary search) and whether the old list holds it already
//   index_merge_kernel  grid over the merged lists: runs of old entries, each shifted by the inserts before it, and the
//                       groups of inserts between them, copied as contiguous pieces
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace siesta {

constexpr int IT = 256;
constexpr int MAX_BUILD_PAIRS = 32;

struct Index {
    Log* log = nullptr;
    int32_t n_pairs = 0;
    std::vector<int32_t> pair_a, pair_b;
    std::vector<int64_t> off;       // [n_pairs + 1] into d_lists
    int64_t* d_lists = nullptr;     // all posting lists back to back (device)
    bool built = false;             // siesta_index_build / siesta_index_refresh (SeqTable view), not loaded lists
};

// ------------------------------------------------------------------------------------------------ compaction
// flags: u8 [n_rows][n]; out rows start at row_off[row]; counts per row returned in row_cnt.
// a flag counts if it is non-zero (want == 0) or equal to `want`
__device__ __forceinline__ bool flag_set(uint8_t f, int want) { return want ? f == want : f != 0; }

__global__ void __launch_bounds__(IT) flag_count_kernel(const uint8_t* flags, int64_t n, int64_t n_blk, unsigned long long* blk, int want) {
    const int row = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * IT + threadIdx.x;
    const unsigned f = (i < n && flag_set(flags[(int64_t)row * n + i], want)) ? 1u : 0u;
    const unsigned ball = __ballot_sync(0xffffffffu, f);
    __shared__ unsigned s[IT / 32];
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = __popc(ball);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned tot = 0;
        for (int k = 0; k < IT / 32; ++k) tot += s[k];
        blk[(int64_t)row * n_blk + blockIdx.x] = tot;
    }
}

// one block per row: exclusive scan of the row's block counts in place; total into row_cnt[row]
__global__ void __launch_bounds__(1024) row_scan_kernel(unsigned long long* blk, int64_t n_blk, unsigned long long* row_cnt) {
    __shared__ unsigned long long ws[32];
    __shared__ unsigned long long carry_s;
    unsigned long long* row = blk + (int64_t)blockIdx.x * n_blk;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < n_blk; base += 1024) {
        const int64_t i = base + threadIdx.x;
        const unsigned long long v = i < n_blk ? row[i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long y = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += y;
        }
        if (lane == 31) ws[warp] = inc;
        __syncthreads();
        unsigned long long before = 0, all = 0;
        for (int k = 0; k < 32; ++k) {
            if (k < warp) before += ws[k];
            all += ws[k];
        }
        const unsigned long long carry = carry_s;
        if (i < n_blk) row[i] = carry + before + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + all;
        __syncthreads();
    }
    if (threadIdx.x == 0) row_cnt[blockIdx.x] = carry_s;
}

// values[i] (or i itself when values == nullptr) of the flagged elements, in order, to out + row_off[row]
__global__ void __launch_bounds__(IT) flag_write_kernel(const uint8_t* flags, const int64_t* values, int64_t n, int64_t n_blk,
                                                       const unsigned long long* blk, const int64_t* row_off, int64_t* out, int want) {
    const int row = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * IT + threadIdx.x;
    const unsigned f = (i < n && flag_set(flags[(int64_t)row * n + i], want)) ? 1u : 0u;
    const unsigned ball = __ballot_sync(0xffffffffu, f);
    __shared__ unsigned s[IT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s[warp] = __popc(ball);
    __syncthreads();
    if (!f) return;
    unsigned before = 0;
    for (int k = 0; k < warp; ++k) before += s[k];
    const int64_t pos = (int64_t)blk[(int64_t)row * n_blk + blockIdx.x] + before + __popc(ball & ((1u << lane) - 1u));
    out[(row_off ? row_off[row] : 0) + pos] = values ? values[i] : i;
}

// ------------------------------------------------------------------------------------------------ index build
struct PairFlagParams {
    const int64_t* trace_off;
    const int32_t* act;
    const int64_t* work;    // nullptr: row t is trace t; else row i is trace work[i]
    int64_t n_traces;       // rows: the log's traces, or the entries of work
    const int8_t* slot_of;  // [n_act] activity -> scratch slot (0..31) or -1
    int32_t n_act;
    int32_t n_pairs;
    int8_t slot_a[MAX_BUILD_PAIRS], slot_b[MAX_BUILD_PAIRS];
    uint8_t* flags;         // [n_pairs][n_traces]
};

__global__ void __launch_bounds__(IT) pair_flags_kernel(const __grid_constant__ PairFlagParams P) {
    __shared__ uint32_t s_cnt[IT / 32][32], s_first[IT / 32][32], s_last[IT / 32][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long warps_total = (long long)gridDim.x * (IT / 32);
    for (long long t = (long long)blockIdx.x * (IT / 32) + warp; t < P.n_traces; t += warps_total) {
        const long long tr = P.work ? P.work[t] : t;
        const long long lo = P.trace_off[tr], hi = P.trace_off[tr + 1];
        s_cnt[warp][lane] = 0;
        s_first[warp][lane] = 0xffffffffu;
        s_last[warp][lane] = 0;
        __syncwarp();
        for (long long i = lo + lane; i < hi; i += 32) {
            const int x = __ldg(P.act + i);
            const int sl = (x >= 0 && x < P.n_act) ? P.slot_of[x] : -1;
            if (sl >= 0) {
                atomicAdd(&s_cnt[warp][sl], 1u);
                atomicMin(&s_first[warp][sl], (uint32_t)(i - lo));
                atomicMax(&s_last[warp][sl], (uint32_t)(i - lo));
            }
        }
        __syncwarp();
        if (lane < P.n_pairs) {
            const int sa = P.slot_a[lane], sb = P.slot_b[lane];
            bool f = false;
            if (sa >= 0 && sb >= 0) {
                if (sa == sb) f = s_cnt[warp][sa] >= 2;
                else f = s_cnt[warp][sa] && s_cnt[warp][sb] && s_first[warp][sa] < s_last[warp][sb];
            }
            P.flags[(long long)lane * P.n_traces + t] = f ? 1 : 0;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------ intersection
struct HitParams {
    int32_t n_lists;
    const int64_t* lists[MAX_BUILD_PAIRS];
    int64_t start[MAX_BUILD_PAIRS + 1];  // list k owns the flat element range [start[k], start[k + 1])
    int64_t n_traces;
    uint32_t* hit;  // [ceil(n_traces / 4)] words = one byte counter per trace
};

// One thread per element of every list.  Lists are duplicate-free and n_lists <= 32, so a byte never overflows into
// its neighbour; ascending ids make the atomics of a warp fall into a few adjacent words.
__global__ void __launch_bounds__(IT) list_hits_kernel(const __grid_constant__ HitParams P) {
    const int64_t i = (int64_t)blockIdx.x * IT + threadIdx.x;
    if (i >= P.start[P.n_lists]) return;
    int k = 0;
    while (i >= P.start[k + 1]) ++k;
    const int64_t t = __ldg(P.lists[k] + (i - P.start[k]));
    if (t >= 0 && t < P.n_traces) atomicAdd(P.hit + (t >> 2), 1u << (8 * (int)(t & 3)));
}

// union over the OR-expansions: mark the traces whose counter reached `want`, and clear the counters for the next one
__global__ void __launch_bounds__(IT) mark_hits_kernel(uint8_t* hit, uint8_t* mark, int64_t n, int want) {
    const int64_t i = (int64_t)blockIdx.x * IT + threadIdx.x;
    if (i >= n) return;
    if (hit[i] == want) mark[i] = 1;
    hit[i] = 0;
}

// hit[t] = number of the given lists that hold trace t (hit must be zero on entry)
static int count_list_hits(Index* ix, const int32_t* ids, int n, uint32_t* d_hit, cudaStream_t stream) {
    HitParams P;
    std::memset(&P, 0, sizeof(P));
    P.n_lists = n;
    for (int k = 0; k < n; ++k) {
        P.lists[k] = ix->d_lists + ix->off[ids[k]];
        P.start[k + 1] = P.start[k] + (ix->off[ids[k] + 1] - ix->off[ids[k]]);
    }
    P.n_traces = ix->log->n_traces;
    P.hit = d_hit;
    if (P.start[n] > 0) {
        list_hits_kernel<<<(unsigned)((P.start[n] + IT - 1) / IT), IT, 0, stream>>>(P);
        SIESTA_LAUNCHED();
        SIESTA_CUDA_OK(cudaGetLastError());
    }
    return SIESTA_OK;
}

static int compact_rows(cudaStream_t stream, const uint8_t* d_flags, const int64_t* d_values, int64_t n, int n_rows,
                        std::vector<int64_t>& counts, int64_t** d_out_all, std::vector<int64_t>& row_off, int want = 0) {
    const int64_t n_blk = std::max<int64_t>((n + IT - 1) / IT, 1);
    unsigned long long *d_blk = nullptr, *d_cnt = nullptr;
    int64_t* d_off = nullptr;
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_blk, sizeof(unsigned long long) * (size_t)n_blk * n_rows, stream));
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_cnt, sizeof(unsigned long long) * (size_t)n_rows, stream));
    dim3 grid((unsigned)n_blk, (unsigned)n_rows);
    flag_count_kernel<<<grid, IT, 0, stream>>>(d_flags, n, n_blk, d_blk, want);
    SIESTA_LAUNCHED();
    row_scan_kernel<<<n_rows, 1024, 0, stream>>>(d_blk, n_blk, d_cnt);
    SIESTA_LAUNCHED();
    std::vector<unsigned long long> h_cnt((size_t)n_rows);
    SIESTA_CUDA_OK(cudaMemcpyAsync(h_cnt.data(), d_cnt, sizeof(unsigned long long) * (size_t)n_rows, cudaMemcpyDeviceToHost, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    counts.assign((size_t)n_rows, 0);
    row_off.assign((size_t)n_rows + 1, 0);
    for (int r = 0; r < n_rows; ++r) {
        counts[r] = (int64_t)h_cnt[r];
        row_off[r + 1] = row_off[r] + counts[r];
    }
    SIESTA_CUDA_OK(cudaMallocAsync((void**)d_out_all, sizeof(int64_t) * (size_t)std::max<int64_t>(row_off[n_rows], 1), stream));
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_off, sizeof(int64_t) * (size_t)(n_rows + 1), stream));
    SIESTA_CUDA_OK(cudaMemcpyAsync(d_off, row_off.data(), sizeof(int64_t) * (size_t)(n_rows + 1), cudaMemcpyHostToDevice, stream));
    flag_write_kernel<<<grid, IT, 0, stream>>>(d_flags, d_values, n, n_blk, d_blk, d_off, *d_out_all, want);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));  // row_off (host vector) was the source of an async copy
    cudaFreeAsync(d_blk, stream);
    cudaFreeAsync(d_cnt, stream);
    cudaFreeAsync(d_off, stream);
    return SIESTA_OK;
}

// Posting lists of the pairs under the SeqTable view over every trace of L (d_work == nullptr) or over the n_work
// ascending traces d_work lists: list p = row_off[p] .. row_off[p + 1]) of *d_lists, ascending trace indices.
static int build_lists(const char* fn, Log* L, const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs, const int64_t* d_work,
                       int64_t n_work, std::vector<int64_t>& row_off, int64_t** d_lists) {
    cudaStream_t stream = L->ctx->stream;
    // activities mentioned by the pairs -> scratch slots
    std::vector<int8_t> slot_of((size_t)std::max(1, L->n_activities), -1);
    PairFlagParams P;
    std::memset(&P, 0, sizeof(P));
    int n_slots = 0;
    auto slot = [&](int a) -> int {
        if (a < 0 || a >= L->n_activities) return -1;  // activity unknown to the log: empty list
        if (slot_of[a] < 0) slot_of[a] = (int8_t)n_slots++;
        return slot_of[a];
    };
    for (int p = 0; p < n_pairs; ++p) {
        P.slot_a[p] = (int8_t)slot(pair_a[p]);
        P.slot_b[p] = (int8_t)slot(pair_b[p]);
        if (n_slots > 32) {
            set_error(std::string(fn) + ": the pairs of one call may mention at most 32 distinct activities");
            return SIESTA_E_UNSUPPORTED;
        }
    }
    const int64_t n = d_work ? n_work : L->n_traces;
    int8_t* d_slot = nullptr;
    uint8_t* d_flags = nullptr;
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_slot, slot_of.size(), stream));
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_flags, (size_t)std::max<int64_t>(n, 1) * n_pairs, stream));
    SIESTA_CUDA_OK(cudaMemcpyAsync(d_slot, slot_of.data(), slot_of.size(), cudaMemcpyHostToDevice, stream));
    P.trace_off = L->d_trace_off;
    P.act = L->d_act;
    P.work = d_work;
    P.n_traces = n;
    P.slot_of = d_slot;
    P.n_act = L->n_activities;
    P.n_pairs = n_pairs;
    P.flags = d_flags;
    if (n > 0) {
        const int64_t ctas = (n + IT / 32 - 1) / (IT / 32);
        const int grid = (int)std::min<int64_t>(ctas, (int64_t)L->ctx->sm_count * 8);
        pair_flags_kernel<<<grid, IT, 0, stream>>>(P);
        SIESTA_LAUNCHED();
        SIESTA_CUDA_OK(cudaGetLastError());
    }
    std::vector<int64_t> counts;
    int rc = compact_rows(stream, d_flags, d_work, n, n_pairs, counts, d_lists, row_off);
    cudaFreeAsync(d_slot, stream);
    cudaFreeAsync(d_flags, stream);
    return rc;
}

// ------------------------------------------------------------------------------------------------ index merge
// The old lists O (back to back) and the delta lists (back to back, same pair order) merge into one flat pass: a delta
// element of pair p that O does not hold goes before O[R] with R = old_off[p] + (its rank in old list p).  Numbered in
// delta order, the k-th such insert lands at R_k + k; R_k never decreases (pairs in order, ranks ascend inside a pair), so
// the output is O cut at the R_k, old run k (between inserts k - 1 and k) shifted by k, with the inserts between the runs.
constexpr int64_t IM_TILE = 8192;   // output entries per block of index_merge_kernel

// One thread per delta element: R[i], nd[i] = 1 unless the old list holds the element, dup[p] += duplicates of pair p.
__global__ void __launch_bounds__(IT) index_dup_kernel(const int64_t* __restrict__ delta, int64_t D, const int64_t* __restrict__ doff,
                                                       int32_t n_pairs, const int64_t* __restrict__ old, const int64_t* __restrict__ ooff,
                                                       int64_t* __restrict__ R, uint8_t* __restrict__ nd, unsigned long long* dup) {
    const int64_t i = (int64_t)blockIdx.x * IT + threadIdx.x;
    int p = 0;
    bool is_dup = false;
    if (i < D) {
        int lo = 0, hi = n_pairs - 1;   // the pair whose delta range holds i: first p with doff[p + 1] > i
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(doff + mid + 1) <= i) lo = mid + 1; else hi = mid;
        }
        p = lo;
        const int64_t x = __ldg(delta + i), end = __ldg(ooff + p + 1);
        int64_t a = __ldg(ooff + p), b = end;
        if (a < b && __ldg(old + b - 1) < x) {
            a = b;   // past the last old entry: every new trace lands here without a search
        } else {
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                if (__ldg(old + mid) < x) a = mid + 1; else b = mid;
            }
        }
        is_dup = a < end && __ldg(old + a) == x;
        R[i] = a;
        nd[i] = is_dup ? 0 : 1;
    }
    const unsigned m = __ballot_sync(0xffffffffu, is_dup);
    if (is_dup) {   // one atomic per pair and warp
        const unsigned same = __match_any_sync(m, p);
        if ((int)(threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(dup + p, (unsigned long long)__popc(same));
    }
}

// Grid over the N merged entries, IM_TILE per block; insert k (value ins[k]) sits at R[k] + k, strictly ascending.  The
// block finds the first insert at or after its tile by binary search, then walks the pieces of the tile: old runs, and
// groups of inserts that share R (no old entry between them) as one contiguous copy.
__global__ void __launch_bounds__(AP_T) index_merge_kernel(const int64_t* __restrict__ old, const int64_t* __restrict__ R,
                                                           const int64_t* __restrict__ ins, int64_t K, int64_t N, int64_t* __restrict__ out) {
    const int64_t o0 = (int64_t)blockIdx.x * IM_TILE;
    const int64_t o1 = o0 + IM_TILE < N ? o0 + IM_TILE : N;
    int64_t lo = 0, hi = K;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (R[mid] + mid < o0) lo = mid + 1; else hi = mid;
    }
    int64_t i = lo, o = o0;   // o is an old entry before insert i, or insert i itself
    while (o < o1) {
        const int64_t d = i < K ? R[i] + i : N;   // old run i ends where insert i sits
        if (o < d) {
            const int64_t n = (d < o1 ? d : o1) - o;
            ap_copy(out + o, old + (o - i), n);
            o += n;
        }
        if (o >= o1 || i >= K) break;
        const int64_t r = R[i];
        int64_t a = i + 1, b = i + (o1 - o) < K ? i + (o1 - o) : K;   // inserts i .. j-1 share r; the tile holds o1 - o
        while (a < b) {
            const int64_t mid = (a + b) >> 1;
            if (R[mid] == r) a = mid + 1; else b = mid;
        }
        const int64_t n = a - i;
        ap_copy(out + o, ins + i, n);
        o += n;
        i = a;
    }
}

// out list p = old list p UNION delta list p (both ascending, duplicate-free); delta lists on the device, offsets on the host.
static int merge_lists(cudaStream_t stream, const int64_t* d_old, const std::vector<int64_t>& old_off, const int64_t* d_delta,
                       const std::vector<int64_t>& doff, int32_t n_pairs, int64_t** d_out, std::vector<int64_t>& new_off) {
    const int64_t D = doff[n_pairs], n_old = old_off[n_pairs];
    std::vector<unsigned long long> h_dup((size_t)n_pairs, 0);
    int64_t *d_doff = nullptr, *d_ooff = nullptr, *d_R = nullptr, *d_insR = nullptr, *d_insV = nullptr;
    unsigned long long *d_dup = nullptr, *d_blk = nullptr, *d_cnt = nullptr;
    uint8_t* d_nd = nullptr;
    const int64_t n_blk = std::max<int64_t>((D + IT - 1) / IT, 1);
    auto release = [&]() {
        for (void* p : {(void*)d_doff, (void*)d_ooff, (void*)d_R, (void*)d_insR, (void*)d_insV, (void*)d_dup, (void*)d_blk, (void*)d_cnt, (void*)d_nd})
            if (p) cudaFreeAsync(p, stream);
    };
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMallocAsync(p, std::max<size_t>(bytes, 8), stream);
    };
    A((void**)&d_doff, sizeof(int64_t) * (size_t)(n_pairs + 1));
    A((void**)&d_ooff, sizeof(int64_t) * (size_t)(n_pairs + 1));
    A((void**)&d_R, sizeof(int64_t) * (size_t)D);
    A((void**)&d_insR, sizeof(int64_t) * (size_t)D);
    A((void**)&d_insV, sizeof(int64_t) * (size_t)D);
    A((void**)&d_nd, (size_t)D);
    A((void**)&d_dup, sizeof(unsigned long long) * (size_t)n_pairs);
    A((void**)&d_blk, sizeof(unsigned long long) * (size_t)n_blk);
    A((void**)&d_cnt, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_doff, doff.data(), sizeof(int64_t) * (size_t)(n_pairs + 1), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ooff, old_off.data(), sizeof(int64_t) * (size_t)(n_pairs + 1), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_dup, 0, sizeof(unsigned long long) * (size_t)n_pairs, stream);
    if (e == cudaSuccess && D > 0) {
        index_dup_kernel<<<(unsigned)n_blk, IT, 0, stream>>>(d_delta, D, d_doff, n_pairs, d_old, d_ooff, d_R, d_nd, d_dup);
        SIESTA_LAUNCHED();
        // inserts in delta order: their R and their values, compacted by the flag scan of the compaction
        flag_count_kernel<<<(unsigned)n_blk, IT, 0, stream>>>(d_nd, D, n_blk, d_blk, 0);
        SIESTA_LAUNCHED();
        row_scan_kernel<<<1, 1024, 0, stream>>>(d_blk, n_blk, d_cnt);
        SIESTA_LAUNCHED();
        flag_write_kernel<<<(unsigned)n_blk, IT, 0, stream>>>(d_nd, d_R, D, n_blk, d_blk, nullptr, d_insR, 0);
        SIESTA_LAUNCHED();
        flag_write_kernel<<<(unsigned)n_blk, IT, 0, stream>>>(d_nd, d_delta, D, n_blk, d_blk, nullptr, d_insV, 0);
        SIESTA_LAUNCHED();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_dup.data(), d_dup, sizeof(unsigned long long) * (size_t)n_pairs, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        release();
        set_error(std::string("index merge: ") + cudaGetErrorString(e));
        return SIESTA_E_CUDA;
    }
    new_off.assign((size_t)n_pairs + 1, 0);
    for (int p = 0; p < n_pairs; ++p)
        new_off[p + 1] = new_off[p] + (old_off[p + 1] - old_off[p]) + (doff[p + 1] - doff[p]) - (int64_t)h_dup[p];
    const int64_t N = new_off[n_pairs], K = N - n_old;
    *d_out = nullptr;
    e = cudaMallocAsync((void**)d_out, sizeof(int64_t) * (size_t)std::max<int64_t>(N, 1), stream);
    if (e == cudaSuccess && N > 0) {
        index_merge_kernel<<<(unsigned)((N + IM_TILE - 1) / IM_TILE), AP_T, 0, stream>>>(d_old, d_insR, d_insV, K, N, *d_out);
        SIESTA_LAUNCHED();
        e = cudaGetLastError();
    }
    release();
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (*d_out) cudaFreeAsync(*d_out, stream);
        *d_out = nullptr;
        set_error(std::string("index merge: ") + cudaGetErrorString(e));
        return SIESTA_E_CUDA;
    }
    return SIESTA_OK;
}

}  // namespace siesta

using namespace siesta;

extern "C" int siesta_index_build(siesta_log* log, const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs,
                                  siesta_index** out) {
    if (!log || !pair_a || !pair_b || !out || n_pairs < 1) {
        set_error("siesta_index_build: bad argument");
        return SIESTA_E_INVALID;
    }
    if (n_pairs > MAX_BUILD_PAIRS) {
        set_error("siesta_index_build: at most " + std::to_string(MAX_BUILD_PAIRS) + " pairs per call");
        return SIESTA_E_UNSUPPORTED;
    }
    Log* L = reinterpret_cast<Log*>(log);
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    Index* ix = new Index();
    ix->log = L;
    ix->n_pairs = n_pairs;
    ix->pair_a.assign(pair_a, pair_a + n_pairs);
    ix->pair_b.assign(pair_b, pair_b + n_pairs);
    ix->built = true;
    int rc = build_lists("siesta_index_build", L, pair_a, pair_b, n_pairs, nullptr, 0, ix->off, &ix->d_lists);
    if (rc) {
        delete ix;
        return rc;
    }
    *out = reinterpret_cast<siesta_index*>(ix);
    return SIESTA_OK;
}

extern "C" int siesta_index_load(siesta_log* log, int32_t n_pairs, const int32_t* pair_a, const int32_t* pair_b,
                                 const int64_t* post_off, const int64_t* trace_idx, siesta_index** out) {
    if (!log || n_pairs < 1 || !pair_a || !pair_b || !post_off || !out || post_off[0] != 0) {
        set_error("siesta_index_load: bad argument");
        return SIESTA_E_INVALID;
    }
    Log* L = reinterpret_cast<Log*>(log);
    for (int p = 0; p < n_pairs; ++p) {
        if (post_off[p + 1] < post_off[p]) {
            set_error("siesta_index_load: post_off must be non-decreasing");
            return SIESTA_E_INVALID;
        }
        for (int64_t i = post_off[p]; i < post_off[p + 1]; ++i)
            if (trace_idx[i] < 0 || trace_idx[i] >= L->n_traces || (i > post_off[p] && trace_idx[i] <= trace_idx[i - 1])) {
                set_error("siesta_index_load: posting lists must be strictly ascending trace indices of this log");
                return SIESTA_E_INVALID;
            }
    }
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    Index* ix = new Index();
    ix->log = L;
    ix->n_pairs = n_pairs;
    ix->pair_a.assign(pair_a, pair_a + n_pairs);
    ix->pair_b.assign(pair_b, pair_b + n_pairs);
    ix->off.assign(post_off, post_off + n_pairs + 1);
    const int64_t total = post_off[n_pairs];
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&ix->d_lists, sizeof(int64_t) * (size_t)std::max<int64_t>(total, 1), L->ctx->stream));
    if (total) SIESTA_CUDA_OK(cudaMemcpyAsync(ix->d_lists, trace_idx, sizeof(int64_t) * (size_t)total, cudaMemcpyHostToDevice, L->ctx->stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(L->ctx->stream));
    *out = reinterpret_cast<siesta_index*>(ix);
    return SIESTA_OK;
}

extern "C" void siesta_index_free(siesta_index* index) {
    if (!index) return;
    Index* ix = reinterpret_cast<Index*>(index);
    cudaSetDevice(ix->log->ctx->device);
    if (ix->d_lists) cudaFreeAsync(ix->d_lists, ix->log->ctx->stream);
    delete ix;
}

extern "C" int64_t siesta_index_list_len(const siesta_index* index, int32_t pair) {
    const Index* ix = reinterpret_cast<const Index*>(index);
    if (!ix || pair < 0 || pair >= ix->n_pairs) return -1;
    return ix->off[pair + 1] - ix->off[pair];
}

extern "C" int siesta_index_get_list(const siesta_index* index, int32_t pair, int64_t* out, int64_t cap) {
    const Index* ix = reinterpret_cast<const Index*>(index);
    if (!ix || pair < 0 || pair >= ix->n_pairs || !out) {
        set_error("siesta_index_get_list: bad argument");
        return SIESTA_E_INVALID;
    }
    const int64_t n = ix->off[pair + 1] - ix->off[pair];
    if (cap < n) {
        set_error("siesta_index_get_list: buffer too small");
        return SIESTA_E_INVALID;
    }
    SIESTA_CUDA_OK(cudaSetDevice(ix->log->ctx->device));
    if (n) SIESTA_CUDA_OK(cudaMemcpyAsync(out, ix->d_lists + ix->off[pair], sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, ix->log->ctx->stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(ix->log->ctx->stream));
    return SIESTA_OK;
}

// result stays on the device (ascending trace indices); free with siesta_device_free
namespace {
// events and stream-ordered scratch of one call, released on every return path
struct CallScratch {
    cudaStream_t s;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    std::vector<void*> bufs;
    explicit CallScratch(cudaStream_t stream) : s(stream) {}
    ~CallScratch() {
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        for (void* p : bufs) cudaFreeAsync(p, s);
    }
    cudaError_t alloc(void** p, size_t bytes) {
        const cudaError_t e = cudaMallocAsync(p, bytes, s);
        if (e == cudaSuccess) bufs.push_back(*p);
        return e;
    }
};
}  // namespace

extern "C" int siesta_intersect_device(siesta_index* index, const int32_t* pair_ids, int32_t n, int64_t** d_out, int64_t* out_n,
                                       double* kernel_ms) {
    Index* ix = reinterpret_cast<Index*>(index);
    if (!ix || !pair_ids || n < 1 || n > MAX_BUILD_PAIRS || !d_out || !out_n) {
        set_error("siesta_intersect: bad argument (1.." + std::to_string(MAX_BUILD_PAIRS) + " lists)");
        return SIESTA_E_INVALID;
    }
    for (int k = 0; k < n; ++k)
        if (pair_ids[k] < 0 || pair_ids[k] >= ix->n_pairs) {
            set_error("siesta_intersect: pair id out of range");
            return SIESTA_E_INVALID;
        }
    SIESTA_CUDA_OK(cudaSetDevice(ix->log->ctx->device));
    cudaStream_t stream = ix->log->ctx->stream;
    // a list named twice would be counted twice: count each distinct list once
    std::vector<int32_t> ids(pair_ids, pair_ids + n);
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    const int nd = (int)ids.size();
    const int64_t T = ix->log->n_traces;
    const size_t hit_bytes = (size_t)((std::max<int64_t>(T, 1) + 3) / 4) * 4;
    CallScratch cs(stream);
    cudaEvent_t& e0 = cs.e0;
    cudaEvent_t& e1 = cs.e1;
    SIESTA_CUDA_OK(cudaEventCreate(&e0));
    SIESTA_CUDA_OK(cudaEventCreate(&e1));
    SIESTA_CUDA_OK(cudaEventRecord(e0, stream));
    uint32_t* d_hit = nullptr;
    SIESTA_CUDA_OK(cs.alloc((void**)&d_hit, hit_bytes));
    SIESTA_CUDA_OK(cudaMemsetAsync(d_hit, 0, hit_bytes, stream));
    int rc = count_list_hits(ix, ids.data(), nd, d_hit, stream);
    std::vector<int64_t> counts, row_off;
    if (rc == SIESTA_OK) rc = compact_rows(stream, reinterpret_cast<const uint8_t*>(d_hit), nullptr, T, 1, counts, d_out, row_off, nd);
    SIESTA_CUDA_OK(cudaEventRecord(e1, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rc) return rc;
    *out_n = counts[0];
    if (kernel_ms) *kernel_ms = ms;
    return SIESTA_OK;
}

extern "C" int siesta_candidates_device(siesta_index* index, const int32_t* exp_off, const int32_t* pair_ids, int32_t n_exp,
                                        int64_t** d_out, int64_t* out_n, double* kernel_ms) {
    Index* ix = reinterpret_cast<Index*>(index);
    if (!ix || !exp_off || !pair_ids || n_exp < 1 || !d_out || !out_n) {
        set_error("siesta_candidates: bad argument");
        return SIESTA_E_INVALID;
    }
    for (int x = 0; x < n_exp; ++x) {
        const int n = exp_off[x + 1] - exp_off[x];
        if (n < 1 || n > MAX_BUILD_PAIRS) {
            set_error("siesta_candidates: every expansion needs 1.." + std::to_string(MAX_BUILD_PAIRS) + " true pairs "
                      "(patterns without a true pair take the Single plan: verify all traces)");
            return SIESTA_E_INVALID;
        }
        for (int k = exp_off[x]; k < exp_off[x + 1]; ++k)
            if (pair_ids[k] < 0 || pair_ids[k] >= ix->n_pairs) {
                set_error("siesta_candidates: pair id out of range");
                return SIESTA_E_INVALID;
            }
    }
    SIESTA_CUDA_OK(cudaSetDevice(ix->log->ctx->device));
    cudaStream_t stream = ix->log->ctx->stream;
    const int64_t T = ix->log->n_traces;
    CallScratch cs(stream);
    cudaEvent_t& e0 = cs.e0;
    cudaEvent_t& e1 = cs.e1;
    SIESTA_CUDA_OK(cudaEventCreate(&e0));
    SIESTA_CUDA_OK(cudaEventCreate(&e1));
    SIESTA_CUDA_OK(cudaEventRecord(e0, stream));
    uint8_t* d_mark = nullptr;
    uint32_t* d_hit = nullptr;
    const size_t hit_bytes = (size_t)((std::max<int64_t>(T, 1) + 3) / 4) * 4;
    SIESTA_CUDA_OK(cs.alloc((void**)&d_mark, (size_t)std::max<int64_t>(T, 1)));
    SIESTA_CUDA_OK(cudaMemsetAsync(d_mark, 0, (size_t)std::max<int64_t>(T, 1), stream));
    SIESTA_CUDA_OK(cs.alloc((void**)&d_hit, hit_bytes));
    SIESTA_CUDA_OK(cudaMemsetAsync(d_hit, 0, hit_bytes, stream));
    for (int x = 0; x < n_exp; ++x) {
        std::vector<int32_t> ids(pair_ids + exp_off[x], pair_ids + exp_off[x + 1]);
        std::sort(ids.begin(), ids.end());
        ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
        int rcx = count_list_hits(ix, ids.data(), (int)ids.size(), d_hit, stream);
        if (rcx) return rcx;
        if (T > 0) {
            mark_hits_kernel<<<(unsigned)((T + IT - 1) / IT), IT, 0, stream>>>(reinterpret_cast<uint8_t*>(d_hit), d_mark, T, (int)ids.size());
            SIESTA_LAUNCHED();
            SIESTA_CUDA_OK(cudaGetLastError());
        }
    }
    std::vector<int64_t> counts, row_off;
    int rc = compact_rows(stream, d_mark, nullptr, T, 1, counts, d_out, row_off);
    SIESTA_CUDA_OK(cudaEventRecord(e1, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rc) return rc;
    *out_n = counts[0];
    if (kernel_ms) *kernel_ms = ms;
    return SIESTA_OK;
}

extern "C" int siesta_candidates(siesta_index* index, const int32_t* exp_off, const int32_t* pair_ids, int32_t n_exp, int64_t* out,
                                 int64_t cap, int64_t* out_n) {
    if (!out_n || (cap && !out)) {
        set_error("siesta_candidates: null output");
        return SIESTA_E_INVALID;
    }
    int64_t* d = nullptr;
    int rc = siesta_candidates_device(index, exp_off, pair_ids, n_exp, &d, out_n, nullptr);
    if (rc) return rc;
    Index* ix = reinterpret_cast<Index*>(index);
    if (*out_n > cap) {
        set_error("siesta_candidates: output buffer too small");
        rc = SIESTA_E_INVALID;
    } else if (*out_n) {
        cudaError_t e = cudaMemcpyAsync(out, d, sizeof(int64_t) * (size_t)*out_n, cudaMemcpyDeviceToHost, ix->log->ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ix->log->ctx->stream);
        if (e != cudaSuccess) {
            set_error(std::string("siesta_candidates: D2H: ") + cudaGetErrorString(e));
            rc = SIESTA_E_CUDA;
        }
    }
    cudaFreeAsync(d, ix->log->ctx->stream);
    return rc;
}

extern "C" void siesta_device_free(siesta_log* log, void* d_ptr) {
    if (!log || !d_ptr) return;
    Log* L = reinterpret_cast<Log*>(log);
    cudaSetDevice(L->ctx->device);
    cudaFreeAsync(d_ptr, L->ctx->stream);
}

extern "C" int siesta_intersect(siesta_index* index, const int32_t* pair_ids, int32_t n, int64_t* out, int64_t cap, int64_t* out_n) {
    if (!out || !out_n) {
        set_error("siesta_intersect: null output");
        return SIESTA_E_INVALID;
    }
    int64_t* d = nullptr;
    int rc = siesta_intersect_device(index, pair_ids, n, &d, out_n, nullptr);
    if (rc) return rc;
    Index* ix = reinterpret_cast<Index*>(index);
    if (*out_n > cap) {
        set_error("siesta_intersect: output buffer too small");
        rc = SIESTA_E_INVALID;
    } else if (*out_n) {
        cudaError_t e = cudaMemcpyAsync(out, d, sizeof(int64_t) * (size_t)*out_n, cudaMemcpyDeviceToHost, ix->log->ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ix->log->ctx->stream);
        if (e != cudaSuccess) {
            set_error(std::string("siesta_intersect: D2H: ") + cudaGetErrorString(e));
            rc = SIESTA_E_CUDA;
        }
    }
    cudaFreeAsync(d, ix->log->ctx->stream);
    return rc;
}

// ------------------------------------------------------------------------------------------------ index after a log append
namespace {
// the new log may carry an index of `ix`'s log: same context, no fewer traces (sets the error)
bool index_log_ok(const char* fn, const Index* ix, const Log* L) {
    if (L->ctx != ix->log->ctx) {
        set_error(std::string(fn) + ": new_log is on another context than the index");
        return false;
    }
    if (L->n_traces < ix->log->n_traces) {
        set_error(std::string(fn) + ": new_log has fewer traces than the index's log");
        return false;
    }
    return true;
}

// *out = a new index on L with ix's pairs and the lists d_lists / off
int finish_index(const Index* ix, Log* L, int64_t* d_lists, std::vector<int64_t>& off, bool built, siesta_index** out) {
    Index* nx = new Index();
    nx->log = L;
    nx->n_pairs = ix->n_pairs;
    nx->pair_a = ix->pair_a;
    nx->pair_b = ix->pair_b;
    nx->off.swap(off);
    nx->d_lists = d_lists;
    nx->built = built;
    *out = reinterpret_cast<siesta_index*>(nx);
    return SIESTA_OK;
}
}  // namespace

extern "C" int siesta_index_append(siesta_index* index, siesta_log* new_log, const int64_t* delta_off, const int64_t* delta_trace_idx,
                                   siesta_index** out, double* kernel_ms) {
    Index* ix = reinterpret_cast<Index*>(index);
    Log* L = reinterpret_cast<Log*>(new_log);
    if (!ix || !L || !delta_off || !out) {
        set_error("siesta_index_append: null argument");
        return SIESTA_E_INVALID;
    }
    if (!index_log_ok("siesta_index_append", ix, L)) return SIESTA_E_INVALID;
    const int32_t n_pairs = ix->n_pairs;
    if (delta_off[0] != 0) {
        set_error("siesta_index_append: delta_off[0] must be 0");
        return SIESTA_E_INVALID;
    }
    for (int p = 0; p < n_pairs; ++p)
        if (delta_off[p + 1] < delta_off[p]) {
            set_error("siesta_index_append: delta_off must be non-decreasing");
            return SIESTA_E_INVALID;
        }
    const int64_t D = delta_off[n_pairs];
    if (D > 0 && !delta_trace_idx) {
        set_error("siesta_index_append: null delta_trace_idx");
        return SIESTA_E_INVALID;
    }
    for (int p = 0; p < n_pairs; ++p)
        for (int64_t i = delta_off[p]; i < delta_off[p + 1]; ++i)
            if (delta_trace_idx[i] < 0 || delta_trace_idx[i] >= L->n_traces || (i > delta_off[p] && delta_trace_idx[i] <= delta_trace_idx[i - 1])) {
                set_error("siesta_index_append: delta lists must be strictly ascending trace indices of new_log");
                return SIESTA_E_INVALID;
            }
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    cudaStream_t stream = L->ctx->stream;
    CallScratch cs(stream);
    int64_t* d_delta = nullptr;
    SIESTA_CUDA_OK(cs.alloc((void**)&d_delta, sizeof(int64_t) * (size_t)std::max<int64_t>(D, 1)));
    if (D) SIESTA_CUDA_OK(cudaMemcpyAsync(d_delta, delta_trace_idx, sizeof(int64_t) * (size_t)D, cudaMemcpyHostToDevice, stream));
    SIESTA_CUDA_OK(cudaEventCreate(&cs.e0));
    SIESTA_CUDA_OK(cudaEventCreate(&cs.e1));
    SIESTA_CUDA_OK(cudaEventRecord(cs.e0, stream));
    std::vector<int64_t> doff(delta_off, delta_off + n_pairs + 1), off;
    int64_t* d_lists = nullptr;
    int rc = merge_lists(stream, ix->d_lists, ix->off, d_delta, doff, n_pairs, &d_lists, off);
    if (rc) return rc;
    cudaError_t e = cudaEventRecord(cs.e1, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, cs.e0, cs.e1);
    if (e != cudaSuccess) {
        cudaFreeAsync(d_lists, stream);
        set_error(std::string("siesta_index_append: ") + cudaGetErrorString(e));
        return SIESTA_E_CUDA;
    }
    if (kernel_ms) *kernel_ms = ms;
    return finish_index(ix, L, d_lists, off, false, out);
}

extern "C" int siesta_index_refresh(siesta_index* index, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed,
                                    siesta_index** out, double* kernel_ms) {
    Index* ix = reinterpret_cast<Index*>(index);
    Log* L = reinterpret_cast<Log*>(new_log);
    if (!ix || !L || !out || n_listed < 0 || (n_listed > 0 && !trace_idx)) {
        set_error("siesta_index_refresh: null argument");
        return SIESTA_E_INVALID;
    }
    if (!ix->built) {
        set_error("siesta_index_refresh: a loaded index cannot be re-derived on the device (use siesta_index_append)");
        return SIESTA_E_INVALID;
    }
    if (!index_log_ok("siesta_index_refresh", ix, L)) return SIESTA_E_INVALID;
    const int64_t T = ix->log->n_traces, T2 = L->n_traces;
    int64_t n_new = 0;
    for (int64_t i = 0; i < n_listed; ++i) {
        if (trace_idx[i] < 0 || trace_idx[i] >= T2 || (i > 0 && trace_idx[i] <= trace_idx[i - 1])) {
            set_error("siesta_index_refresh: trace_idx must ascend strictly inside [0, new_log's n_traces)");
            return SIESTA_E_INVALID;
        }
        n_new += trace_idx[i] >= T;
    }
    if (n_new != T2 - T) {
        set_error("siesta_index_refresh: trace_idx must list every trace new_log adds (as passed to siesta_log_append)");
        return SIESTA_E_INVALID;
    }
    // Ids outside the old log's alphabet that the new alphabet covers: when a pair names one, unlisted traces may hold it
    // and gain the pair, so every trace is flagged again.
    bool all = false;
    if (!ix->log->act_valid)
        for (int p = 0; p < ix->n_pairs; ++p)
            for (int32_t a : {ix->pair_a[p], ix->pair_b[p]})
                all |= a >= ix->log->n_activities && a < L->n_activities;
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    cudaStream_t stream = L->ctx->stream;
    CallScratch cs(stream);
    int64_t* d_work = nullptr;
    if (!all) {
        SIESTA_CUDA_OK(cs.alloc((void**)&d_work, sizeof(int64_t) * (size_t)std::max<int64_t>(n_listed, 1)));
        if (n_listed) SIESTA_CUDA_OK(cudaMemcpyAsync(d_work, trace_idx, sizeof(int64_t) * (size_t)n_listed, cudaMemcpyHostToDevice, stream));
    }
    SIESTA_CUDA_OK(cudaEventCreate(&cs.e0));
    SIESTA_CUDA_OK(cudaEventCreate(&cs.e1));
    SIESTA_CUDA_OK(cudaEventRecord(cs.e0, stream));
    std::vector<int64_t> doff, off;
    int64_t *d_delta = nullptr, *d_lists = nullptr;
    int rc = build_lists("siesta_index_refresh", L, ix->pair_a.data(), ix->pair_b.data(), ix->n_pairs, all ? nullptr : d_work, n_listed,
                         all ? off : doff, all ? &d_lists : &d_delta);
    if (rc) return rc;
    if (!all) {
        rc = merge_lists(stream, ix->d_lists, ix->off, d_delta, doff, ix->n_pairs, &d_lists, off);
        cudaFreeAsync(d_delta, stream);
        if (rc) return rc;
    }
    cudaError_t e = cudaEventRecord(cs.e1, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, cs.e0, cs.e1);
    if (e != cudaSuccess) {
        cudaFreeAsync(d_lists, stream);
        set_error(std::string("siesta_index_refresh: ") + cudaGetErrorString(e));
        return SIESTA_E_CUDA;
    }
    if (kernel_ms) *kernel_ms = ms;
    return finish_index(ix, L, d_lists, off, true, out);
}
