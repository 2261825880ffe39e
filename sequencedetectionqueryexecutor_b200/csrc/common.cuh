// common.cuh — shared host/device declarations of libsiesta_gpu (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/siesta_gpu.h"

namespace siesta {

void set_error(const std::string& msg);
struct Ctx;
// a block of at least `bytes` from the context's device arena (nullptr: out of memory, error set); a block may be
// returned only when no kernel uses it any more (the callers return blocks after they have waited for their stream)
void* dev_arena_alloc(Ctx* c, size_t bytes);
void dev_arena_free(Ctx* c, void* p);
// owner record behind siesta_dev_matches::impl
struct DevMatchesImpl {
    void* block = nullptr;
    Ctx* owner = nullptr;
};
extern std::atomic<long long> g_kernel_launches;

#define SIESTA_CUDA_OK(expr)                                                                      \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            ::siesta::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
            return SIESTA_E_CUDA;                                                                 \
        }                                                                                         \
    } while (0)

#define SIESTA_LAUNCHED() (::siesta::g_kernel_launches.fetch_add(1, std::memory_order_relaxed))

// Block-wide copy of n elements by blocks of AP_T threads (append.cu, intersect.cu).  16-byte loads and stores when
// source and destination agree modulo 16 bytes (scalar head and tail), coalesced element copies otherwise.
constexpr int AP_T = 256;
#ifdef __CUDACC__
template <typename T>
__device__ __forceinline__ void ap_copy(T* __restrict__ dst, const T* __restrict__ src, int64_t n) {
    constexpr int V = 16 / sizeof(T);
    if ((((uintptr_t)dst ^ (uintptr_t)src) & 15) == 0) {
        int64_t head = (int64_t)(((16 - ((uintptr_t)dst & 15)) & 15) / sizeof(T));
        head = head < n ? head : n;
        if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
        const int64_t nv = (n - head) / V;
        int4* __restrict__ dv = reinterpret_cast<int4*>(dst + head);
        const int4* __restrict__ sv = reinterpret_cast<const int4*>(src + head);
#pragma unroll 4
        for (int64_t i = threadIdx.x; i < nv; i += AP_T) dv[i] = __ldg(sv + i);
        const int64_t done = head + nv * V;
        if (done + threadIdx.x < n) dst[done + threadIdx.x] = src[done + threadIdx.x];
    } else {
#pragma unroll 8
        for (int64_t i = threadIdx.x; i < n; i += AP_T) dst[i] = __ldg(src + i);
    }
}
#endif

// Pinned host blocks that result objects (siesta_matches) are carved from; blocks return here on siesta_matches_free
// and are reused by later calls, so a steady-state request pays no cudaHostAlloc.
struct HostBlock {
    void* p;
    size_t size;
    bool used;
};

// Device blocks that requests take their scratch and their results from; blocks return here and are reused by later
// requests, so a steady-state request performs no device allocation at all.  (Stream-ordered cudaMallocAsync was
// measured to stall a request for ~13 ms now and then - one in ten to forty requests on an 8-GPU run, when a 0.7 GB
// scratch block and a 2.4 GB result alternate in the pool - which is four times the request itself.)
struct DevBlock {
    void* p;
    size_t size;
    bool used;
};

struct Ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    std::mutex arena_mu;
    std::vector<HostBlock> arena;
    std::vector<unsigned long long*> pinned_counters;  // free 128-byte pinned blocks for the requests' counters ...
    std::vector<DevBlock> dev_arena;                   // guarded by arena_mu
    std::vector<void*> pinned_slabs;                   // ... carved from slabs of 32 (one cudaHostAlloc each: the call may wait
                                                       // for running kernels, and a request in flight may be spinning on a peer)
};

// CSR event log resident in HBM.
struct Log {
    Ctx* ctx = nullptr;
    const int64_t* d_trace_off = nullptr;  // [T+1]
    const int32_t* d_act = nullptr;        // [E]
    const int64_t* d_ts_ms = nullptr;      // [E]
    const int64_t* d_src_event = nullptr;  // [E] derived logs (logview.cu): index of the event in the source log
    int64_t n_traces = 0, n_events = 0;
    int32_t n_activities = 0;
    int32_t max_trace_len = 0;             // caller's hint (wrapped logs) or exact (loaded logs)
    int64_t true_max_len = -1;             // exact, measured on the device on first use (declare counting); -1 = not yet
    bool owns = false;
    int64_t first_trace = 0;  // global index of trace 0 (multi-GPU shards)
    // Block-cyclic shard (siesta_log_set_blocks): local traces [blk_local[b], blk_local[b + 1]) are the global traces
    // starting at blk_global[b].  n_blocks == 0: one contiguous range starting at first_trace.
    int32_t n_blocks = 0;
    int64_t blk_local[SIESTA_MAX_BLOCKS + 1] = {0};
    int64_t blk_global[SIESTA_MAX_BLOCKS] = {0};
    bool act_valid = false;  // every activity id lies in [0, n_activities): kernels may skip the per-event range check
};

// Device-side NFA: SIESTA's State[] flattened (S/query/State.java, AdditionalState.java).
struct DevNfa {
    int32_t n_states;
    uint32_t init_st;   // Run.initializeRun: negative -> 2, kleeneClosure* -> 3 (S/engine/Run.java:146-155), 2 bits/state
    uint32_t all2;      // st field of a complete run: every state == 2 (Run.checkMatch, Run.java:181-191)
    uint8_t kind[SIESTA_MAX_STATES];
    uint8_t n_preds[SIESTA_MAX_STATES];
    uint8_t has_vv;     // bit k: some predicate references state k (NFA.hasValueVector, S/query/NFA.java:462-469)
    uint8_t need_vv;
    uint8_t any_kleene;
    uint8_t merge_safe;  // dominated-run merging is exact for this NFA (see validate_nfa)
    uint8_t cross_safe;  // ... also across value-vector families (all predicates reference earlier states)
    uint8_t fast_class;  // FAST_* (detect_fast.cuh): the NFA and the flags admit a closed-form evaluator
    int8_t kmax[SIESTA_MAX_STATES + 1];                 // largest slot a run at state c can still read, -1 = none
    unsigned long long relmask[SIESTA_MAX_STATES + 1];  // byte k = 0xFF iff a predicate of a state >= c references state k
    uint8_t p_attr[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];
    uint8_t p_op[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];
    uint8_t p_ref[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];
    int64_t p_c[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];
};

// Window-walk program of an NK-class NFA for kernel K1-P (derivation: detect_fast.cuh), built by nkw_build (nfa.cpp),
// which also decides the index space the masks live in (NKW_NONE: the NFA stays on the staged kernel).
enum { NKW_NONE = 0, NKW_RANK = 1, NKW_RAW = 2 };

struct NkwProgram {
    int32_t n_states;
    uint8_t neg[SIESTA_MAX_STATES];                      // state k is a negative state
    uint8_t n_preds[SIESTA_MAX_STATES];
    uint8_t le[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];     // 1: e below bit idx(ref) + cc, 0: e at or above it
    uint8_t sh[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];     // 8 * referenced state (byte of the packed indices)
    uint8_t cc[SIESTA_MAX_STATES][SIESTA_MAX_PREDS];     // min(c, 64) (+ 1 for <=)
    // Markov form (every predicate of a positive state references the positive state before it; a negative state in
    // between carries no predicate and neither does the state after it): all starts are evaluated at once, backwards
    // (nkw_markov, detect_fast.cuh).  For positive state k >= 1: prev[k] = the positive state before it, m_ge[k] / m_le[k] =
    // the event taken for k lies between ge and le index steps after the one taken for prev[k] (le = 255: unbounded).
    uint8_t markov;
    uint8_t prev[SIESTA_MAX_STATES], m_ge[SIESTA_MAX_STATES], m_le[SIESTA_MAX_STATES];
};

int nkw_build(const DevNfa& dn, uint32_t flags, NkwProgram* out);

struct DetectPending;
// Chunked evaluation (siesta_evaluate_events): where a chunk's results sit in the whole result.
struct RebaseOffsets {
    int64_t trace, occ, ev;
};
int detect_device_impl(Log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand, uint32_t flags, cudaStream_t stream,
                       RebaseOffsets base, siesta_dev_matches* out);
int validate_act_range(Log* L, int64_t first_event, int64_t n_events, cudaStream_t stream);
// Host checks of an appended batch against a log of T traces (siesta_log_append's rules; sets the error, append.cu)
bool append_check_batch(const char* fn, int64_t T, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                        const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces);
// K3 refresh after a log append on one log (declare.cu; siesta_multi_declare_counts_refresh runs it on every shard)
struct DeclareRefresh {
    Log* O = nullptr;                  // the log before the append (only read)
    Log* N = nullptr;                  // the log after it
    int64_t n_listed = 0, n_old = 0;   // listed traces; those below O's n_traces (a prefix of the ascending list)
    int64_t* d_work = nullptr;         // the listed traces on the device (in `block`)
    int64_t max_old = 0, max_new = 0;  // longest listed trace in O / N (measured for pair-kernel alphabets only)
    void* block = nullptr;             // arena blocks, returned by declare_refresh_release
    void* scratch = nullptr;
};
// host checks (null trace_idx, k_cap, contexts, derived or blocked logs, shrinking logs, trace_idx; sets the error)
bool declare_refresh_check_host(const char* fn, const Log* O, const Log* N, const int64_t* trace_idx, int64_t n_listed, int32_t k_cap);
bool declare_refresh_needs_full(const Log* O, const Log* N);
// listed traces to the device (`copied`, may be null, is recorded after the copy) + the device check of the unlisted traces'
// lengths (SIESTA_E_INVALID) + pair widths; waits
int declare_refresh_stage(const char* fn, DeclareRefresh* r, const int64_t* trace_idx, cudaStream_t stream, cudaEvent_t copied);
// d_delta (N's layout) = K3(N, listed) - K3(O, listed old traces); enqueues only
int declare_refresh_delta(DeclareRefresh* r, int32_t k_cap, int64_t* d_delta, cudaStream_t stream);
// d_out = d_old moved from alphabet A0 to A1 + d_delta (d_out may be d_delta, or d_old when A0 == A1); enqueues only
int declare_merge(const int64_t* d_old, int32_t A0, int32_t A1, int32_t k_cap, const int64_t* d_delta, int64_t* d_out, const Ctx* c,
                  cudaStream_t stream);
void declare_refresh_release(DeclareRefresh* r, cudaStream_t stream);
int assemble_matches(Ctx* c, std::vector<siesta_dev_matches>& parts, uint32_t flags, cudaStream_t stream, siesta_matches** out,
                     const std::vector<Ctx*>* part_ctx);
int detect_device_finish_impl(DetectPending* q, siesta_dev_matches* out);
void detect_pending_set_base(DetectPending* q, RebaseOffsets base);

int validate_nfa(const siesta_nfa* nfa, uint32_t flags, DevNfa* out);

// ------------------------------------------------------------------------------------------ multi-GPU exchange (multi.cu)
// Header of a rank's compact result block in its exchange region (wire format: multi.cu).  Written on the device when
// the block is complete; every rank reads every header (sizes travel in-band: no size collective, no host round trip
// before the payload moves).
constexpr int XCHG_MAX_RANKS = 16;
constexpr size_t XCHG_CTRL_BYTES = 8192;   // control pages at the start of a region; the data area follows
constexpr int64_t XCHG_ERR_CAP = 4096;     // error / outlier list entries a block carries
enum { XST_LIMITS = 1, XST_STAGING = 2, XST_RANGE = 4, XST_ERRCAP = 8, XST_TIMEOUT = 16 };
struct XHeader {
    unsigned long long seq;
    int64_t n_tr, n_occ, n_ev, n_err, n_emitted, n_unsup;
    int64_t trace_base;        // global index of the shard's first trace
    int32_t all_cols, seconds; // event columns present; ts_delta in seconds (EventTs route) or milliseconds
    int32_t uniform_k;         // > 0: one occurrence per trace and uniform_k events per occurrence (no offset sections)
    int32_t status;            // XST_* bits: the request failed on this rank
    int64_t o_trace, o_base, o_occ_off, o_ev_off, o_pos, o_rank, o_act, o_delta, o_err, o_unsup;   // byte offsets into the block
    int64_t slot_off;          // byte offset of the block inside the rank's data area (one slot per block of a blocked log)
    int64_t shard_traces;      // traces of the rank's whole shard (all blocks): the capacity the receivers plan with
    int64_t pad[10];
};
static_assert(sizeof(XHeader) == 256, "XHeader is 256 bytes");
// Where the placement writes the compact block (detect.cu: detect_device_pack_impl)
struct PackTarget {
    char* data;            // data area of the local exchange region
    int64_t cap_bytes;
    XHeader* hdr;          // header slot of the local region
    unsigned long long seq;
    int64_t slot_off = 0;      // -> XHeader::slot_off
    int64_t shard_traces = 0;  // -> XHeader::shard_traces
};
int detect_device_begin_impl(Log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand, uint32_t flags,
                             cudaStream_t stream, RebaseOffsets base, DetectPending** pending, const DetectPending* sibling = nullptr);
int detect_device_pack_impl(DetectPending* q, const PackTarget& tgt);   // enqueues only, no host wait
void detect_pending_discard(DetectPending* q);
float detect_pending_k1_ms(DetectPending* q);                            // releases the request (stream-ordered)
int64_t detect_pack_required_bytes(int64_t n_cand_or_traces, int64_t n_events_log, int uniform_k, bool all_cols, bool return_all);
int detect_uniform_k(const siesta_nfa* nfa, uint32_t flags);
bool detect_nkp_eligible(const siesta_nfa* nfa, uint32_t flags, int32_t n_activities);
void build_lut(const siesta_nfa* nfa, const DevNfa& dn, int32_t n_activities, uint32_t flags, std::vector<uint16_t>& lut,
               int* needs_ts, int* n_positive);

}  // namespace siesta
