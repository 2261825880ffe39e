// multi.cu — the multi-GPU exchange of libsiesta_gpu: match lists joined by a device-side all-gather, counts by a
// device-side all-reduce, both over NVLink peer memory, both behind the C-ABI (include/siesta_gpu.h, siesta_exchange_*).
//
// The reference has no counterpart (it is one JVM with Spark local[*]); the path it stands behind is
// QueryPlanPatternDetection.execute (J/model/Queries/QueryPlans/Detection/QueryPlanPatternDetection.java:106-131), whose
// SaseConnector.evaluate loop over ALL candidate traces is what the shards split.
//
// One exchange object per rank (GPU).  A rank owns ONE device region, [control page | data area], that every peer maps:
// across processes through a CUDA IPC handle (siesta_exchange_export / _import: one process per GPU, e.g. under
// torchrun), inside one process through peer access (siesta_exchange_connect_local: one JVM driving all GPUs).
// A collective operation (every rank calls them in the same order) is numbered `seq` and runs as
//   wait    until every peer has acknowledged pulling operation seq - 1 out of my region        (xchg_wait_acks_kernel)
//   produce my block INTO my region: the placement of the match list (detect.cu, gather_packed_kernel) with the sizes
//           in the block's header, or the count array
//   signal  st.release.sys `seq` into every peer's ready slot; wait for every peer's; fetch their headers
//                                                                                                 (xchg_signal_kernel)
//   pull    read every peer's block over NVLink and, in the same kernel, decode it to the standard columns at its
//           place in the joined list (xchg_decode_*_kernel) / reduce the count arrays in rank order (xchg_reduce_kernel)
//   ack     st.release.sys `seq` into every peer's ack slot                                       (xchg_ack_kernel)
// No size collective, no host round trip before the payload moves: the host waits once for the headers (it needs the
// sizes to allocate the joined result) and once for the end of the request.  Every spin is bounded (XCHG_TIMEOUT_NS):
// a missing peer fails the request, it does not hang the GPU.
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace siesta {

constexpr unsigned long long XCHG_TIMEOUT_NS = 20ull * 1000 * 1000 * 1000;

constexpr int XCHG_MAX_BLOCKS = SIESTA_MAX_BLOCKS;
struct XCtrl {
    XHeader hdr[XCHG_MAX_BLOCKS];                // hdr[b]: header of block b of the request in flight (slot 0: every other operation)
    unsigned long long ready[XCHG_MAX_RANKS];    // ready[p]: written by rank p - its block of operation `value` is complete
    unsigned long long ack[XCHG_MAX_RANKS];      // ack[p]:   written by rank p - it has pulled my blocks up to operation `value`
};
static_assert(sizeof(XCtrl) <= XCHG_CTRL_BYTES, "control pages");

struct XPeers {
    char* region[XCHG_MAX_RANKS];
};

// Places of one block's ranks in the joined list (absolute exclusive prefixes) and the running totals of a request; both
// live in device memory and are advanced by xchg_prefix_kernel block by block, so a block is decoded as soon as every
// rank has announced it - no host round trip per block.
struct XBases {
    int64_t tb[XCHG_MAX_RANKS + 1], ob[XCHG_MAX_RANKS + 1], eb[XCHG_MAX_RANKS + 1], rb[XCHG_MAX_RANKS + 1], ub[XCHG_MAX_RANKS + 1];
};
struct XRun {
    int64_t n_tr, n_occ, n_ev, n_err, n_unsup, n_emitted;
    int32_t status;       // OR of the headers' status bits (and XST_TIMEOUT for a block that is out of step)
    int32_t pad;
};
struct XDev {
    XHeader hdrs[XCHG_MAX_BLOCKS * XCHG_MAX_RANKS];   // [block][rank], as fetched by the wait kernels
    XBases bases[XCHG_MAX_BLOCKS];
    XRun run;
    int flag;                                         // a device-side wait timed out
    int pad[15];
};

struct Exchange {
    Ctx* ctx = nullptr;
    int world = 1, rank = 0;
    char* region = nullptr;
    size_t cap_bytes = 0;
    XPeers peers;
    bool ipc[XCHG_MAX_RANKS];
    bool connected[XCHG_MAX_RANKS];
    unsigned long long seq = 0;
    cudaStream_t stream = nullptr;    // scan, placement, announcements
    cudaStream_t jstream = nullptr;   // waits for the peers, pulls + decodes (higher priority: its CTAs go first when SMs free up)
    XDev* d_x = nullptr;
    XDev* h_x = nullptr;              // pinned copy
    std::mutex mu;                    // one collective at a time per exchange
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// spins until *p >= want; false on timeout
__device__ __forceinline__ bool spin_until(const unsigned long long* p, unsigned long long want) {
    const unsigned long long t0 = global_ns();
    while (ld_acquire_sys(p) < want) {
        if (global_ns() - t0 > XCHG_TIMEOUT_NS) return false;
        __nanosleep(200);
    }
    return true;
}

__global__ void xchg_wait_acks_kernel(XCtrl* me, int world, int rank, unsigned long long seq_prev, int* timed_out) {
    const int p = threadIdx.x;
    if (p < world && p != rank && !spin_until(&me->ack[p], seq_prev)) atomicOr(timed_out, 1);
}

// announce: my block of operation `seq` is complete (everything the kernels before this one wrote is visible first)
__global__ void xchg_post_kernel(const __grid_constant__ XPeers peers, int world, int rank, unsigned long long seq) {
    const int p = threadIdx.x;
    if (p >= world) return;
    __threadfence_system();
    st_release_sys(&reinterpret_cast<XCtrl*>(peers.region[p])->ready[rank], seq);
}

// wait until every rank has announced operation `seq`, then fetch header slot `slot` of every rank into d_hdrs[0..world)
__global__ void xchg_wait_kernel(const __grid_constant__ XPeers peers, int world, int rank, unsigned long long seq, int slot, XHeader* d_hdrs,
                                 int* timed_out) {
    const int p = threadIdx.x;
    if (p >= world) return;
    const bool ok = spin_until(&reinterpret_cast<XCtrl*>(peers.region[rank])->ready[p], seq);
    XHeader h;
    if (ok) {
        const volatile uint4* src = reinterpret_cast<const volatile uint4*>(&reinterpret_cast<XCtrl*>(peers.region[p])->hdr[slot]);
        uint4* dst = reinterpret_cast<uint4*>(&h);
#pragma unroll
        for (int i = 0; i < (int)(sizeof(XHeader) / 16); ++i) {
            uint4 v;
            v.x = src[i].x; v.y = src[i].y; v.z = src[i].z; v.w = src[i].w;
            dst[i] = v;
        }
        if (!h.status && h.seq != seq) {   // the peer is out of step (another request, another number of blocks)
            memset(&h, 0, sizeof(h));
            h.status = XST_TIMEOUT;
        }
    } else {
        memset(&h, 0, sizeof(h));
        h.status = XST_TIMEOUT;
        atomicOr(timed_out, 1);
    }
    d_hdrs[p] = h;
}

// announce + wait + fetch in one launch (the count all-reduce: one block, nothing to overlap)
__global__ void xchg_signal_kernel(const __grid_constant__ XPeers peers, int world, int rank, unsigned long long seq, XHeader* d_hdrs,
                                   int* timed_out) {
    const int p = threadIdx.x;
    if (p >= world) return;
    __threadfence_system();   // the block written by the kernels before this one is visible system-wide before the flag
    st_release_sys(&reinterpret_cast<XCtrl*>(peers.region[p])->ready[rank], seq);
    const bool ok = spin_until(&reinterpret_cast<XCtrl*>(peers.region[rank])->ready[p], seq);
    XHeader h;
    if (ok) {
        const volatile uint4* src = reinterpret_cast<const volatile uint4*>(&reinterpret_cast<XCtrl*>(peers.region[p])->hdr[0]);
        uint4* dst = reinterpret_cast<uint4*>(&h);
#pragma unroll
        for (int i = 0; i < (int)(sizeof(XHeader) / 16); ++i) {
            uint4 v;
            v.x = src[i].x; v.y = src[i].y; v.z = src[i].z; v.w = src[i].w;
            dst[i] = v;
        }
    } else {
        memset(&h, 0, sizeof(h));
        h.status = XST_TIMEOUT;
        atomicOr(timed_out, 1);
    }
    d_hdrs[p] = h;
}

__global__ void xchg_ack_kernel(const __grid_constant__ XPeers peers, int world, int rank, unsigned long long seq) {
    const int p = threadIdx.x;
    if (p >= world) return;
    __threadfence_system();
    st_release_sys(&reinterpret_cast<XCtrl*>(peers.region[p])->ack[rank], seq);
}

// places of block `blk`'s ranks in the joined list: the running totals so far + the sizes in the block's headers
__global__ void xchg_prefix_kernel(XDev* d, int blk, int world) {
    if (threadIdx.x || blockIdx.x) return;
    XRun run = d->run;
    XBases& B = d->bases[blk];
    const XHeader* h = d->hdrs + blk * XCHG_MAX_RANKS;
    B.tb[0] = run.n_tr; B.ob[0] = run.n_occ; B.eb[0] = run.n_ev; B.rb[0] = run.n_err; B.ub[0] = run.n_unsup;
    for (int p = 0; p < world; ++p) {
        const bool good = h[p].status == 0;
        run.status |= h[p].status;
        B.tb[p + 1] = B.tb[p] + (good ? h[p].n_tr : 0);
        B.ob[p + 1] = B.ob[p] + (good ? h[p].n_occ : 0);
        B.eb[p + 1] = B.eb[p] + (good ? h[p].n_ev : 0);
        B.rb[p + 1] = B.rb[p] + (good ? h[p].n_err : 0);
        B.ub[p + 1] = B.ub[p] + (good ? h[p].n_unsup : 0);
        run.n_emitted += good ? h[p].n_emitted : 0;
    }
    run.n_tr = B.tb[world]; run.n_occ = B.ob[world]; run.n_ev = B.eb[world]; run.n_err = B.rb[world]; run.n_unsup = B.ub[world];
    d->run = run;
}

// ------------------------------------------------------------------------------------------------ pull + decode
struct XDecode {
    int world, me;   // grid row y handles source rank (me + y) % world: at any moment the ranks read from different peers
    const char* data[XCHG_MAX_RANKS];   // data areas of all ranks (mine included)
    const XHeader* hdrs;                // [world] headers of the block, device copy
    const XBases* bases;                // the ranks' places in the joined list (device memory: xchg_prefix_kernel)
    int64_t *trace_idx, *occ_off, *ev_off;
    int32_t *pos, *rank, *act;
    int64_t* ts;
    int64_t* err;
    int64_t* unsup;
};

// Uniform blocks (one occurrence per trace, K events per occurrence): a CTA takes tiles of TE events of one rank.  The
// tile's four event sections come in with 16-byte loads (whole lines over NVLink), are widened out of shared memory and
// leave as coalesced 4- and 8-byte stores at the rank's place in the joined list.
constexpr int XD_THREADS = 256;
constexpr int XD_TE = 2048;
__global__ void __launch_bounds__(XD_THREADS) xchg_decode_uniform_kernel(const __grid_constant__ XDecode D) {
    __shared__ __align__(16) uint16_t s_pos[XD_TE];
    __shared__ __align__(16) uint8_t s_rank[XD_TE];
    __shared__ __align__(16) uint16_t s_act[XD_TE];
    __shared__ __align__(16) int32_t s_delta[XD_TE];
    __shared__ long long s_base[XD_TE + 1];
    const int r = (int)((blockIdx.y + D.me) % D.world);
    const XHeader h = D.hdrs[r];
    if (h.status) return;
    const int K = h.uniform_k;
    const char* data = D.data[r] + h.slot_off;
    const int tid = threadIdx.x;
    const int64_t n_ev = h.n_ev, n_tr = h.n_tr;
    const int64_t eb = D.bases->eb[r], tb = D.bases->tb[r];
    const long long unit = h.seconds ? 1000 : 1;
    const uint32_t* g_trace = reinterpret_cast<const uint32_t*>(data + h.o_trace);
    const long long* g_base = reinterpret_cast<const long long*>(data + h.o_base);
    for (int64_t e0 = (int64_t)blockIdx.x * XD_TE; e0 < n_ev; e0 += (int64_t)gridDim.x * XD_TE) {
        const int cnt = (int)min((int64_t)XD_TE, n_ev - e0);
        // 16-byte chunks that hold at least one event of the tile (sections are 256-byte aligned and e0 is a multiple
        // of 2048: aligned; a chunk may end past n_ev: still inside the section's capacity)
        {
            const uint4* gp = reinterpret_cast<const uint4*>(data + h.o_pos) + e0 / 8;
            if (tid * 8 < cnt) reinterpret_cast<uint4*>(s_pos)[tid] = __ldcv(gp + tid);
            if (h.all_cols) {
                const uint4* gr = reinterpret_cast<const uint4*>(data + h.o_rank) + e0 / 16;
                const uint4* ga = reinterpret_cast<const uint4*>(data + h.o_act) + e0 / 8;
                const uint4* gd = reinterpret_cast<const uint4*>(data + h.o_delta) + e0 / 4;
                if (tid * 16 < cnt) reinterpret_cast<uint4*>(s_rank)[tid] = __ldcv(gr + tid);
                if (tid * 8 < cnt) reinterpret_cast<uint4*>(s_act)[tid] = __ldcv(ga + tid);
                if (tid * 4 < cnt) reinterpret_cast<uint4*>(s_delta)[tid] = __ldcv(gd + tid);
                if ((tid + XD_THREADS) * 4 < cnt) reinterpret_cast<uint4*>(s_delta)[tid + XD_THREADS] = __ldcv(gd + tid + XD_THREADS);
                const int64_t t0 = e0 / K, t1 = (e0 + cnt - 1) / K;   // traces that own the tile's events
                for (int64_t t = t0 + tid; t <= t1; t += XD_THREADS) s_base[t - t0] = __ldcv(g_base + t);
            }
        }
        __syncthreads();
        {
            // event i of the tile belongs to trace (r0 + i) / K of the tile (r0 = events of the tile's first trace that sit
            // in the previous tile): small numbers, so the division is one multiply-high by ceil(2^32 / K)
            const uint32_t r0 = (uint32_t)(e0 - (e0 / K) * K);
            const uint32_t magic = (uint32_t)((0x100000000ull + (unsigned)K - 1) / (unsigned)K);
            int32_t* o_pos = D.pos + eb + e0;
            int32_t* o_rank = h.all_cols ? D.rank + eb + e0 : nullptr;
            int32_t* o_act = h.all_cols ? D.act + eb + e0 : nullptr;
            long long* o_ts = h.all_cols ? reinterpret_cast<long long*>(D.ts) + eb + e0 : nullptr;
#pragma unroll 4
            for (int i = tid; i < cnt; i += XD_THREADS) {
                o_pos[i] = (int32_t)s_pos[i];
                if (h.all_cols) {
                    o_rank[i] = (int32_t)s_rank[i];
                    o_act[i] = (int32_t)s_act[i];
                    o_ts[i] = s_base[K == 1 ? (r0 + i) : __umulhi(r0 + (uint32_t)i, magic)] + (long long)s_delta[i] * unit;
                }
            }
        }
        __syncthreads();
    }
    for (int64_t t = (int64_t)blockIdx.x * XD_THREADS + tid; t < n_tr; t += (int64_t)gridDim.x * XD_THREADS) {
        D.trace_idx[tb + t] = h.trace_base + (int64_t)__ldcv(g_trace + t);
        D.occ_off[tb + t] = tb + t;            // one occurrence per trace: occurrence index == trace index
        D.ev_off[tb + t] = eb + t * K;
    }
    for (int64_t i = (int64_t)blockIdx.x * XD_THREADS + tid; i < h.n_err; i += (int64_t)gridDim.x * XD_THREADS)
        D.err[D.bases->rb[r] + i] = h.trace_base + __ldcv(reinterpret_cast<const long long*>(data + h.o_err) + i);
    for (int64_t i = (int64_t)blockIdx.x * XD_THREADS + tid; i < h.n_unsup; i += (int64_t)gridDim.x * XD_THREADS)
        D.unsup[D.bases->ub[r] + i] = h.trace_base + __ldcv(reinterpret_cast<const long long*>(data + h.o_unsup) + i);
}

// General blocks (any number of occurrences per trace and of events per occurrence): one thread per trace.
__global__ void __launch_bounds__(XD_THREADS) xchg_decode_general_kernel(const __grid_constant__ XDecode D) {
    const int r = (int)((blockIdx.y + D.me) % D.world);
    const XHeader h = D.hdrs[r];
    if (h.status) return;
    const char* data = D.data[r] + h.slot_off;
    const uint32_t* g_trace = reinterpret_cast<const uint32_t*>(data + h.o_trace);
    const long long* g_base = reinterpret_cast<const long long*>(data + h.o_base);
    const uint32_t* g_occ = reinterpret_cast<const uint32_t*>(data + h.o_occ_off);
    const uint32_t* g_evo = reinterpret_cast<const uint32_t*>(data + h.o_ev_off);
    const uint16_t* g_pos = reinterpret_cast<const uint16_t*>(data + h.o_pos);
    const uint8_t* g_rank = reinterpret_cast<const uint8_t*>(data + h.o_rank);
    const uint16_t* g_act = reinterpret_cast<const uint16_t*>(data + h.o_act);
    const int32_t* g_delta = reinterpret_cast<const int32_t*>(data + h.o_delta);
    const int64_t tb = D.bases->tb[r], ob = D.bases->ob[r], eb = D.bases->eb[r];
    const long long unit = h.seconds ? 1000 : 1;
    for (int64_t t = (int64_t)blockIdx.x * XD_THREADS + threadIdx.x; t < h.n_tr; t += (int64_t)gridDim.x * XD_THREADS) {
        D.trace_idx[tb + t] = h.trace_base + (int64_t)__ldcv(g_trace + t);
        const int64_t o0 = __ldcv(g_occ + t), o1 = __ldcv(g_occ + t + 1);
        D.occ_off[tb + t] = ob + o0;
        const long long base = h.all_cols ? __ldcv(g_base + t) : 0;
        for (int64_t o = o0; o < o1; ++o) {
            const int64_t a = __ldcv(g_evo + o), b = __ldcv(g_evo + o + 1);
            D.ev_off[ob + o] = eb + a;
            for (int64_t e = a; e < b; ++e) {
                D.pos[eb + e] = (int32_t)__ldcv(g_pos + e);
                if (h.all_cols) {
                    D.rank[eb + e] = (int32_t)__ldcv(g_rank + e);
                    D.act[eb + e] = (int32_t)__ldcv(g_act + e);
                    D.ts[eb + e] = base + (long long)__ldcv(g_delta + e) * unit;
                }
            }
        }
    }
    for (int64_t i = (int64_t)blockIdx.x * XD_THREADS + threadIdx.x; i < h.n_err; i += (int64_t)gridDim.x * XD_THREADS)
        D.err[D.bases->rb[r] + i] = h.trace_base + __ldcv(reinterpret_cast<const long long*>(data + h.o_err) + i);
    for (int64_t i = (int64_t)blockIdx.x * XD_THREADS + threadIdx.x; i < h.n_unsup; i += (int64_t)gridDim.x * XD_THREADS)
        D.unsup[D.bases->ub[r] + i] = h.trace_base + __ldcv(reinterpret_cast<const long long*>(data + h.o_unsup) + i);
}

__global__ void xchg_tail_kernel(int64_t* occ_off, int64_t* ev_off, const XRun* run) {
    occ_off[run->n_tr] = run->n_occ;
    ev_off[run->n_occ] = run->n_ev;
}

// all-reduce of int64 arrays that sit at the start of every rank's data area: out[i] = op over the ranks, in rank order
__global__ void xchg_reduce_kernel(const __grid_constant__ XPeers peers, int world, int64_t n, int op, int64_t* out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        long long acc = __ldcv(reinterpret_cast<const long long*>(peers.region[0] + XCHG_CTRL_BYTES) + i);
        for (int p = 1; p < world; ++p) {
            const long long v = __ldcv(reinterpret_cast<const long long*>(peers.region[p] + XCHG_CTRL_BYTES) + i);
            acc = op == SIESTA_REDUCE_SUM ? acc + v : (op == SIESTA_REDUCE_MIN ? (v < acc ? v : acc) : (v > acc ? v : acc));
        }
        out[i] = acc;
    }
}

static int check_ready(Exchange* x, const char* who) {
    if (!x) {
        set_error(std::string(who) + ": null exchange");
        return SIESTA_E_INVALID;
    }
    for (int p = 0; p < x->world; ++p)
        if (!x->connected[p]) {
            set_error(std::string(who) + ": rank " + std::to_string(p) + " is not connected (siesta_exchange_import / _connect_local)");
            return SIESTA_E_INVALID;
        }
    return SIESTA_OK;
}

}  // namespace siesta

using namespace siesta;

extern "C" int siesta_exchange_create(siesta_ctx* ctx, int32_t world, int32_t rank, int64_t capacity_bytes, siesta_exchange** out) {
    if (!ctx || !out || world < 1 || world > XCHG_MAX_RANKS || rank < 0 || rank >= world || capacity_bytes < 0) {
        set_error("siesta_exchange_create: bad argument (1 <= world <= 16, 0 <= rank < world)");
        return SIESTA_E_INVALID;
    }
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    SIESTA_CUDA_OK(cudaSetDevice(c->device));
    Exchange* x = new Exchange();
    x->ctx = c;
    x->world = world;
    x->rank = rank;
    x->cap_bytes = ((size_t)capacity_bytes + 255) & ~(size_t)255;
    std::memset(&x->peers, 0, sizeof(x->peers));
    std::memset(x->ipc, 0, sizeof(x->ipc));
    std::memset(x->connected, 0, sizeof(x->connected));
    // plain cudaMalloc: IPC handles cannot be taken of stream-ordered pool memory
    cudaError_t e = cudaMalloc((void**)&x->region, XCHG_CTRL_BYTES + x->cap_bytes);
    if (e != cudaSuccess) {
        set_error(std::string("siesta_exchange_create: cudaMalloc(") + std::to_string(XCHG_CTRL_BYTES + x->cap_bytes) + "): " + cudaGetErrorString(e));
        delete x;
        return SIESTA_E_NOMEM;
    }
    e = cudaMemset(x->region, 0, XCHG_CTRL_BYTES);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        int lo = 0, hi = 0;   // (lowest, greatest) priority; greatest is numerically smallest
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        const char* env = std::getenv("SIESTA_XCHG_JOIN_PRIORITY");   // tuning aid: "low" = the join's CTAs yield to the scan's
        e = cudaStreamCreateWithPriority(&x->jstream, cudaStreamNonBlocking, env && env[0] == 'l' ? lo : hi);
    }
    if (e == cudaSuccess) {
        // Load every kernel and driver-internal copy path a collective uses NOW: with lazy module loading the first
        // launch of a function may wait for the device to drain, and inside a collective another rank of this process
        // may already be spinning on this one (ranks that share a device in the tests; one JVM driving all GPUs).
        cudaFuncAttributes fa;
        cudaFuncGetAttributes(&fa, xchg_wait_acks_kernel);
        cudaFuncGetAttributes(&fa, xchg_signal_kernel);
        cudaFuncGetAttributes(&fa, xchg_post_kernel);
        cudaFuncGetAttributes(&fa, xchg_wait_kernel);
        cudaFuncGetAttributes(&fa, xchg_prefix_kernel);
        cudaFuncGetAttributes(&fa, xchg_ack_kernel);
        cudaFuncGetAttributes(&fa, xchg_decode_uniform_kernel);
        cudaFuncGetAttributes(&fa, xchg_decode_general_kernel);
        cudaFuncGetAttributes(&fa, xchg_tail_kernel);
        cudaFuncGetAttributes(&fa, xchg_reduce_kernel);
        XHeader warm;
        std::memset(&warm, 0, sizeof(warm));
        cudaMemcpyAsync(x->region, &warm, sizeof(warm), cudaMemcpyHostToDevice, x->stream);
        cudaMemcpyAsync(x->region + XCHG_CTRL_BYTES, x->region, std::min<size_t>(256, x->cap_bytes), cudaMemcpyDeviceToDevice, x->stream);
        cudaMemsetAsync(x->region + XCHG_CTRL_BYTES, 0, std::min<size_t>(256, x->cap_bytes), x->stream);
        xchg_reduce_kernel<<<1, 32, 0, x->stream>>>(x->peers, 0, 0, SIESTA_REDUCE_SUM, nullptr);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_x, sizeof(XDev));
    if (e == cudaSuccess) e = cudaMemset(x->d_x, 0, sizeof(XDev));
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&x->h_x, sizeof(XDev), cudaHostAllocDefault);
    if (e == cudaSuccess) {
        std::memset(x->h_x, 0, sizeof(XDev));
        xchg_prefix_kernel<<<1, 32, 0, x->jstream>>>(x->d_x, 0, 0);
        xchg_tail_kernel<<<1, 1, 0, x->jstream>>>(reinterpret_cast<int64_t*>(x->region + XCHG_CTRL_BYTES),
                                                  reinterpret_cast<int64_t*>(x->region + XCHG_CTRL_BYTES), &x->d_x->run);
        e = cudaMemcpyAsync(x->h_x, x->d_x, sizeof(XDev), cudaMemcpyDeviceToHost, x->jstream);
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error(std::string("siesta_exchange_create: ") + cudaGetErrorString(e));
        siesta_exchange_free(reinterpret_cast<siesta_exchange*>(x));
        return SIESTA_E_CUDA;
    }
    x->peers.region[rank] = x->region;
    x->connected[rank] = true;
    *out = reinterpret_cast<siesta_exchange*>(x);
    return SIESTA_OK;
}

extern "C" int siesta_exchange_export(siesta_exchange* xh, void* handle_out) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    if (!x || !handle_out) {
        set_error("siesta_exchange_export: null argument");
        return SIESTA_E_INVALID;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == SIESTA_EXCHANGE_HANDLE_BYTES, "IPC handle size");
    SIESTA_CUDA_OK(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    SIESTA_CUDA_OK(cudaIpcGetMemHandle(&h, x->region));
    std::memcpy(handle_out, &h, sizeof(h));
    return SIESTA_OK;
}

extern "C" int siesta_exchange_import(siesta_exchange* xh, int32_t peer_rank, const void* handle) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    if (!x || !handle || peer_rank < 0 || peer_rank >= x->world || peer_rank == x->rank) {
        set_error("siesta_exchange_import: bad argument");
        return SIESTA_E_INVALID;
    }
    SIESTA_CUDA_OK(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    void* p = nullptr;
    SIESTA_CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    x->peers.region[peer_rank] = reinterpret_cast<char*>(p);
    x->ipc[peer_rank] = true;
    x->connected[peer_rank] = true;
    return SIESTA_OK;
}

extern "C" int siesta_exchange_connect_local(siesta_exchange* xh, int32_t peer_rank, siesta_exchange* peer) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    Exchange* y = reinterpret_cast<Exchange*>(peer);
    if (!x || !y || peer_rank < 0 || peer_rank >= x->world || peer_rank == x->rank || y->rank != peer_rank || y->world != x->world) {
        set_error("siesta_exchange_connect_local: bad argument");
        return SIESTA_E_INVALID;
    }
    if (y->ctx->device != x->ctx->device) {
        SIESTA_CUDA_OK(cudaSetDevice(x->ctx->device));
        int can = 0;
        SIESTA_CUDA_OK(cudaDeviceCanAccessPeer(&can, x->ctx->device, y->ctx->device));
        if (!can) {
            set_error("siesta_exchange_connect_local: no peer access between the two devices");
            return SIESTA_E_CUDA;
        }
        const cudaError_t e = cudaDeviceEnablePeerAccess(y->ctx->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
            set_error(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            return SIESTA_E_CUDA;
        }
        cudaGetLastError();
    }
    x->peers.region[peer_rank] = y->region;
    x->connected[peer_rank] = true;
    return SIESTA_OK;
}

extern "C" void siesta_exchange_free(siesta_exchange* xh) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    if (!x) return;
    cudaSetDevice(x->ctx->device);
    if (x->stream) cudaStreamSynchronize(x->stream);
    if (x->jstream) cudaStreamSynchronize(x->jstream);
    for (int p = 0; p < x->world; ++p)
        if (x->ipc[p] && x->peers.region[p]) cudaIpcCloseMemHandle(x->peers.region[p]);
    if (x->region) cudaFree(x->region);
    if (x->d_x) cudaFree(x->d_x);
    if (x->h_x) cudaFreeHost(x->h_x);
    if (x->stream) cudaStreamDestroy(x->stream);
    if (x->jstream) cudaStreamDestroy(x->jstream);
    delete x;
}

// the blocks of a shard log: [first local trace, one past the last), global index of the first trace
static int log_blocks(const Log* L, int64_t (&lo)[XCHG_MAX_BLOCKS], int64_t (&hi)[XCHG_MAX_BLOCKS], int64_t (&glob)[XCHG_MAX_BLOCKS]) {
    if (L->n_blocks <= 0) {
        lo[0] = 0;
        hi[0] = L->n_traces;
        glob[0] = L->first_trace;
        return 1;
    }
    for (int b = 0; b < L->n_blocks; ++b) {
        lo[b] = L->blk_local[b];
        hi[b] = L->blk_local[b + 1];
        glob[b] = L->blk_global[b];
    }
    return L->n_blocks;
}

extern "C" int64_t siesta_exchange_required_bytes(siesta_log* log, const siesta_nfa* nfa, uint32_t flags) {
    Log* L = reinterpret_cast<Log*>(log);
    if (!L || !nfa) return -1;
    int64_t lo[XCHG_MAX_BLOCKS], hi[XCHG_MAX_BLOCKS], glob[XCHG_MAX_BLOCKS];
    const int C = log_blocks(L, lo, hi, glob);
    int64_t need = 0;   // one slot per block: a block stays in the region until every peer has pulled it
    for (int b = 0; b < C; ++b)
        need += detect_pack_required_bytes(hi[b] - lo[b], L->n_events, detect_uniform_k(nfa, flags), !(flags & SIESTA_F_NO_EVENT_COLUMNS),
                                           (flags & SIESTA_F_RETURN_ALL) != 0);
    return need;
}

extern "C" int siesta_detect_allgather(siesta_log* log, const siesta_nfa* nfa, uint32_t flags, siesta_exchange* xh,
                                       siesta_dev_matches* out, siesta_exchange_stats* stats) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    Log* L = reinterpret_cast<Log*>(log);
    if (!L || !nfa || !out) {
        set_error("siesta_detect_allgather: null argument");
        return SIESTA_E_INVALID;
    }
    int rc = check_ready(x, "siesta_detect_allgather");
    if (rc) return rc;
    if (L->ctx != x->ctx) {
        set_error("siesta_detect_allgather: the log and the exchange belong to different contexts");
        return SIESTA_E_INVALID;
    }
    std::memset(out, 0, sizeof(*out));
    if (stats) std::memset(stats, 0, sizeof(*stats));
    std::lock_guard<std::mutex> lock(x->mu);
    SIESTA_CUDA_OK(cudaSetDevice(x->ctx->device));
    const int world = x->world, rank = x->rank;
    XCtrl* me = reinterpret_cast<XCtrl*>(x->region);
    XDev* dx = x->d_x;
    XDev* hx = x->h_x;
    const bool all_cols = !(flags & SIESTA_F_NO_EVENT_COLUMNS);

    // ---- the blocks of my shard (one for a contiguous shard): each is verified, placed and announced on its own, in
    // order, on stream S; operation numbers are consecutive, block b of this request is operation seq0 + 1 + b
    int64_t b_lo[XCHG_MAX_BLOCKS], b_hi[XCHG_MAX_BLOCKS], b_glob[XCHG_MAX_BLOCKS];
    const int C = log_blocks(L, b_lo, b_hi, b_glob);
    // one block: nothing to overlap, the join follows the scan on the same stream
    cudaStream_t S = x->stream, J = (C == 1 && std::getenv("SIESTA_XCHG_TWO_STREAMS") == nullptr) ? x->stream : x->jstream;
    const unsigned long long seq0 = x->seq;
    x->seq += (unsigned long long)C;
    const unsigned long long seq_last = seq0 + (unsigned long long)C;
    std::vector<Log> view((size_t)C, *L);
    int64_t slot_off[XCHG_MAX_BLOCKS], slot_bytes[XCHG_MAX_BLOCKS];
    {
        const int uk = detect_uniform_k(nfa, flags);
        int64_t at = 0;
        for (int b = 0; b < C; ++b) {
            Log& V = view[(size_t)b];
            V.d_trace_off = L->d_trace_off + b_lo[b];   // offsets stay absolute: the event columns are shared
            V.n_traces = b_hi[b] - b_lo[b];
            V.first_trace = b_glob[b];
            V.n_blocks = 0;
            V.owns = false;
            slot_off[b] = at;
            slot_bytes[b] = detect_pack_required_bytes(V.n_traces, L->n_events, uk, all_cols, (flags & SIESTA_F_RETURN_ALL) != 0);
            at += slot_bytes[b];
        }
    }

    enum { EV_S0 = 0, EV_S1, EV_J0, EV_J1, EV_RESET, EV_H0, EV_D0, N_EV };
    cudaEvent_t ev[N_EV] = {nullptr};
    struct EvGuard {
        cudaEvent_t* e;
        ~EvGuard() { for (int i = 0; i < N_EV; ++i) if (e[i]) cudaEventDestroy(e[i]); }
    } ev_guard{ev};
    for (int i = 0; i < N_EV; ++i) SIESTA_CUDA_OK(cudaEventCreate(&ev[i]));
    std::vector<DetectPending*> pend((size_t)C, nullptr);
    struct PendGuard {   // the scans' scratch goes back to the arena once both streams are idle
        std::vector<DetectPending*>& q;
        cudaStream_t a, b;
        ~PendGuard() {
            cudaStreamSynchronize(a);
            cudaStreamSynchronize(b);
            for (DetectPending* p : q) if (p) detect_pending_discard(p);
        }
    } pend_guard{pend, S, J};

    SIESTA_CUDA_OK(cudaMemsetAsync(&dx->run, 0, sizeof(XRun) + sizeof(int), S));   // running totals and the time-out flag
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_RESET], S));
    SIESTA_CUDA_OK(cudaStreamWaitEvent(J, ev[EV_RESET], 0));
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_S0], S));
    std::string first_error;
    for (int b = 0; b < C; ++b) {
        if (!rc) {
            const int rcb = detect_device_begin_impl(&view[(size_t)b], nfa, nullptr, 0, flags, S, RebaseOffsets{0, 0, 0}, &pend[(size_t)b],
                                                     b > 0 ? pend[0] : nullptr);
            if (rcb) {
                rc = rcb;
                first_error = siesta_last_error();
            }
        }
        // my region is rewritten from here on: every peer must have pulled the previous operation's blocks out of it
        if (b == 0) {
            xchg_wait_acks_kernel<<<1, 32, 0, S>>>(me, world, rank, seq0, &dx->flag);
            SIESTA_LAUNCHED();
        }
        int fail = rc ? XST_LIMITS : 0;
        if (!rc) {
            PackTarget tgt{x->region + XCHG_CTRL_BYTES + slot_off[b], std::min<int64_t>(slot_bytes[b], (int64_t)x->cap_bytes - slot_off[b]),
                           &me->hdr[b], seq0 + 1 + (unsigned long long)b};
            tgt.slot_off = slot_off[b];
            tgt.shard_traces = L->n_traces;
            const int rc2 = detect_device_pack_impl(pend[(size_t)b], tgt);
            if (rc2) {
                rc = rc2;
                first_error = siesta_last_error();
                fail = XST_STAGING;
            }
        }
        if (fail) {   // keep the collective in step: the peers wait for this block - announce a failed one
            XHeader fh;
            std::memset(&fh, 0, sizeof(fh));
            fh.seq = seq0 + 1 + (unsigned long long)b;
            fh.status = fail;
            cudaMemcpyAsync(&me->hdr[b], &fh, sizeof(fh), cudaMemcpyHostToDevice, S);
        }
        xchg_post_kernel<<<1, 32, 0, S>>>(x->peers, world, rank, seq0 + 1 + (unsigned long long)b);
        SIESTA_LAUNCHED();
    }
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_S1], S));

    // ---- stream J: block 0 of every rank -> its headers tell how the request continues
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_J0], J));
    xchg_wait_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq0 + 1, 0, dx->hdrs, &dx->flag);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaMemcpyAsync(hx->hdrs, dx->hdrs, sizeof(XHeader) * XCHG_MAX_RANKS, cudaMemcpyDeviceToHost, J));
    SIESTA_CUDA_OK(cudaMemcpyAsync(&hx->flag, &dx->flag, sizeof(int), cudaMemcpyDeviceToHost, J));
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_H0], J));
    SIESTA_CUDA_OK(cudaEventSynchronize(ev[EV_H0]));   // host wait 1 of 2 (my later blocks keep running on S)

    // every rank sees the same headers, so every rank takes the same path from here
    auto finish_failed = [&](int bad, bool skip_waits = false) -> int {
        // all ranks fail this request, and all acknowledge it so that the next one can overwrite the regions; the
        // later blocks are waited for first (bounded) unless a peer is missing already
        if (!(bad & XST_TIMEOUT) && !skip_waits)
            for (int b = 1; b < C; ++b) {
                xchg_wait_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq0 + 1 + (unsigned long long)b, b, dx->hdrs + b * XCHG_MAX_RANKS, &dx->flag);
                SIESTA_LAUNCHED();
            }
        xchg_ack_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq_last);
        SIESTA_LAUNCHED();
        cudaStreamSynchronize(J);
        cudaStreamSynchronize(S);
        if (rc) {
            set_error(first_error);
            return rc;
        }
        if (bad & XST_TIMEOUT) {
            set_error("exchange: a peer did not arrive within the time limit (or is out of step)");
            return SIESTA_E_CUDA;
        }
        if (bad & XST_LIMITS) {
            set_error("exchange: too many traces beyond the engine limits on some rank, or its verification failed (see siesta_detect)");
            return SIESTA_E_UNSUPPORTED;
        }
        if (bad & XST_RANGE) {
            set_error("exchange: a value does not fit the compact block (trace longer than 65 535 events, activity id >= 65 536, "
                      "a timestamp more than 2^31 units from the trace's first reported event)");
            return SIESTA_E_UNSUPPORTED;
        }
        set_error("exchange: staging overflow or too many reference errors on some rank");
        return SIESTA_E_NOMEM;
    };
    int bad = hx->flag ? XST_TIMEOUT : 0;
    bool uniform = true;
    int64_t cap_tr = 0;
    for (int p = 0; p < world; ++p) {
        const XHeader& h = hx->hdrs[p];
        bad |= h.status;
        uniform = uniform && h.uniform_k > 0;
        cap_tr += h.shard_traces;
    }
    if (bad || rc) return finish_failed(bad);
    const int K = uniform ? hx->hdrs[0].uniform_k : 0;

    // ---- the joined result: one allocation, the library's standard columns.  Eager: sized for the worst case now and
    // filled block by block; otherwise sized exactly once the last block's headers are in.
    auto layout = [&](int64_t n_tr, int64_t n_occ, int64_t n_ev, int64_t n_err, int64_t n_unsup, size_t (&q)[9]) {
        size_t f_off = 0;
        auto fcarve = [&f_off](size_t bytes) {
            const size_t at = f_off;
            f_off += (bytes + 255) & ~(size_t)255;
            return at;
        };
        q[0] = fcarve((size_t)n_tr * 8);
        q[1] = fcarve((size_t)(n_tr + 1) * 8);
        q[2] = fcarve((size_t)(n_occ + 1) * 8);
        q[3] = fcarve((size_t)n_ev * 4);
        q[4] = fcarve((size_t)n_err * 8);
        q[5] = q[6] = q[7] = 0;
        if (all_cols) {
            q[5] = fcarve((size_t)n_ev * 4);
            q[6] = fcarve((size_t)n_ev * 4);
            q[7] = fcarve((size_t)n_ev * 8);
        }
        q[8] = fcarve((size_t)n_unsup * 8);
        return f_off;
    };
    size_t qo[9];
    size_t f_bytes = 0;
    bool eager = false;
    if (C > 1 && uniform) {
        const int64_t lists = (int64_t)XCHG_ERR_CAP * world * C;
        f_bytes = layout(cap_tr, cap_tr, cap_tr * K, lists, lists, qo);
        size_t limit = (size_t)24 << 30;
        if (const char* env = std::getenv("SIESTA_XCHG_EAGER_MAX_BYTES")) limit = (size_t)std::strtoull(env, nullptr, 10);
        eager = f_bytes <= limit;
    }
    XDecode D;
    std::memset(&D, 0, sizeof(D));
    D.world = world;
    D.me = rank;
    for (int p = 0; p < world; ++p) D.data[p] = x->peers.region[p] + XCHG_CTRL_BYTES;
    void* fin_owned = nullptr;
    struct FinGuard {   // an error return below gives the block back
        Ctx* c;
        void*& p;
        ~FinGuard() { if (p) dev_arena_free(c, p); }
    } fin_guard{x->ctx, fin_owned};
    auto bind = [&](void* fin) {
        char* fb = reinterpret_cast<char*>(fin);
        D.trace_idx = reinterpret_cast<int64_t*>(fb + qo[0]);
        D.occ_off = reinterpret_cast<int64_t*>(fb + qo[1]);
        D.ev_off = reinterpret_cast<int64_t*>(fb + qo[2]);
        D.pos = reinterpret_cast<int32_t*>(fb + qo[3]);
        D.err = reinterpret_cast<int64_t*>(fb + qo[4]);
        D.rank = all_cols ? reinterpret_cast<int32_t*>(fb + qo[5]) : nullptr;
        D.act = all_cols ? reinterpret_cast<int32_t*>(fb + qo[6]) : nullptr;
        D.ts = all_cols ? reinterpret_cast<int64_t*>(fb + qo[7]) : nullptr;
        D.unsup = reinterpret_cast<int64_t*>(fb + qo[8]);
    };
    // grid of one block's decode: row y = source rank (me + y) % world; columns sized from the largest block
    auto decode_block = [&](int b, int64_t biggest_units) {
        // all rows together stay within ONE wave of resident CTAs (34 KB of shared memory each: six per SM): measured at
        // N = 2, 148 / 296 / 593 / 1184 CTAs per row: 1.79 / 1.06 / 1.49 / 1.16 ms
        int gx = (int)std::min<int64_t>(std::max<int64_t>(biggest_units, 1), std::max(1, x->ctx->sm_count * 4 / world));
        if (const char* env = std::getenv("SIESTA_XCHG_DECODE_CTAS")) {
            const int v = std::atoi(env);
            if (v >= 1) gx = v;
        }
        XDecode Db = D;
        Db.hdrs = dx->hdrs + b * XCHG_MAX_RANKS;
        Db.bases = dx->bases + b;
        xchg_prefix_kernel<<<1, 32, 0, J>>>(dx, b, world);
        SIESTA_LAUNCHED();
        const dim3 grid((unsigned)gx, (unsigned)world);
        if (uniform) xchg_decode_uniform_kernel<<<grid, XD_THREADS, 0, J>>>(Db);
        else xchg_decode_general_kernel<<<grid, XD_THREADS, 0, J>>>(Db);
        SIESTA_LAUNCHED();
    };
    if (eager) {
        fin_owned = dev_arena_alloc(x->ctx, f_bytes);
        if (!fin_owned) {
            first_error = siesta_last_error();
            rc = SIESTA_E_NOMEM;   // (this rank only; it still waits for the blocks and acknowledges them)
            return finish_failed(0);
        }
        bind(fin_owned);
        SIESTA_CUDA_OK(cudaEventRecord(ev[EV_D0], J));
        int64_t big = 1;
        for (int p = 0; p < world; ++p) big = std::max(big, (hx->hdrs[p].shard_traces / C + 1) * K / XD_TE + 1);
        decode_block(0, big);
        for (int b = 1; b < C; ++b) {
            xchg_wait_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq0 + 1 + (unsigned long long)b, b, dx->hdrs + b * XCHG_MAX_RANKS, &dx->flag);
            SIESTA_LAUNCHED();
            decode_block(b, big);
        }
    } else {
        for (int b = 1; b < C; ++b) {
            xchg_wait_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq0 + 1 + (unsigned long long)b, b, dx->hdrs + b * XCHG_MAX_RANKS, &dx->flag);
            SIESTA_LAUNCHED();
        }
        if (C > 1) {
            SIESTA_CUDA_OK(cudaMemcpyAsync(hx->hdrs, dx->hdrs, sizeof(XHeader) * XCHG_MAX_RANKS * (size_t)C, cudaMemcpyDeviceToHost, J));
            SIESTA_CUDA_OK(cudaMemcpyAsync(&hx->flag, &dx->flag, sizeof(int), cudaMemcpyDeviceToHost, J));
            SIESTA_CUDA_OK(cudaStreamSynchronize(J));
            bad = hx->flag ? XST_TIMEOUT : 0;
            for (int b = 0; b < C; ++b)
                for (int p = 0; p < world; ++p) bad |= hx->hdrs[b * XCHG_MAX_RANKS + p].status;
            if (bad) return finish_failed(bad, true);
        }
        int64_t t_tr = 0, t_occ = 0, t_ev = 0, t_err = 0, t_unsup = 0;
        for (int b = 0; b < C; ++b)
            for (int p = 0; p < world; ++p) {
                const XHeader& h = hx->hdrs[b * XCHG_MAX_RANKS + p];
                t_tr += h.n_tr; t_occ += h.n_occ; t_ev += h.n_ev; t_err += h.n_err; t_unsup += h.n_unsup;
            }
        f_bytes = layout(t_tr, t_occ, t_ev, t_err, t_unsup, qo);
        fin_owned = dev_arena_alloc(x->ctx, f_bytes);
        if (!fin_owned) {
            first_error = siesta_last_error();
            rc = SIESTA_E_NOMEM;
            return finish_failed(0, true);
        }
        bind(fin_owned);
        SIESTA_CUDA_OK(cudaEventRecord(ev[EV_D0], J));
        for (int b = 0; b < C; ++b) {
            int64_t big = 1;
            for (int p = 0; p < world; ++p) {
                const XHeader& h = hx->hdrs[b * XCHG_MAX_RANKS + p];
                big = std::max(big, uniform ? h.n_ev / XD_TE + 1 : h.n_tr / XD_THREADS + 1);
            }
            decode_block(b, big);
        }
    }
    xchg_tail_kernel<<<1, 1, 0, J>>>(D.occ_off, D.ev_off, &dx->run);
    SIESTA_LAUNCHED();
    xchg_ack_kernel<<<1, 32, 0, J>>>(x->peers, world, rank, seq_last);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaEventRecord(ev[EV_J1], J));
    SIESTA_CUDA_OK(cudaMemcpyAsync(hx->hdrs, dx->hdrs, sizeof(XHeader) * XCHG_MAX_RANKS * (size_t)C, cudaMemcpyDeviceToHost, J));
    SIESTA_CUDA_OK(cudaMemcpyAsync(&hx->run, &dx->run, sizeof(XRun) + sizeof(int), cudaMemcpyDeviceToHost, J));
    SIESTA_CUDA_OK(cudaStreamSynchronize(J));   // host wait 2 of 2: the joined list is complete on this rank
    SIESTA_CUDA_OK(cudaStreamSynchronize(S));
    const XRun run = hx->run;
    bad = (hx->flag ? XST_TIMEOUT : 0) | run.status;
    if (bad) {   // (already acknowledged)
        rc = SIESTA_OK;
        if (bad & XST_TIMEOUT) {
            set_error("exchange: a peer did not arrive within the time limit (or is out of step)");
            return SIESTA_E_CUDA;
        }
        if (bad & XST_LIMITS) {
            set_error("exchange: too many traces beyond the engine limits on some rank, or its verification failed (see siesta_detect)");
            return SIESTA_E_UNSUPPORTED;
        }
        if (bad & XST_RANGE) {
            set_error("exchange: a value does not fit the compact block (trace longer than 65 535 events, activity id >= 65 536, "
                      "a timestamp more than 2^31 units from the trace's first reported event)");
            return SIESTA_E_UNSUPPORTED;
        }
        set_error("exchange: staging overflow or too many reference errors on some rank");
        return SIESTA_E_NOMEM;
    }
    const int64_t n_tr = run.n_tr, n_occ = run.n_occ, n_ev = run.n_ev, n_err = run.n_err, n_unsup = run.n_unsup;
    if (n_err > 0) {   // the (rare) error list in ascending order
        std::vector<int64_t> herr((size_t)n_err);
        SIESTA_CUDA_OK(cudaMemcpyAsync(herr.data(), D.err, (size_t)n_err * 8, cudaMemcpyDeviceToHost, J));
        SIESTA_CUDA_OK(cudaStreamSynchronize(J));
        std::sort(herr.begin(), herr.end());
        SIESTA_CUDA_OK(cudaMemcpyAsync(D.err, herr.data(), (size_t)n_err * 8, cudaMemcpyHostToDevice, J));
        SIESTA_CUDA_OK(cudaStreamSynchronize(J));
    }
    if (n_unsup > 0) {   // per-rank lists arrive in completion order
        std::vector<int64_t> hu((size_t)n_unsup);
        SIESTA_CUDA_OK(cudaMemcpyAsync(hu.data(), D.unsup, (size_t)n_unsup * 8, cudaMemcpyDeviceToHost, J));
        SIESTA_CUDA_OK(cudaStreamSynchronize(J));
        std::sort(hu.begin(), hu.end());
        SIESTA_CUDA_OK(cudaMemcpyAsync(D.unsup, hu.data(), (size_t)n_unsup * 8, cudaMemcpyHostToDevice, J));
        SIESTA_CUDA_OK(cudaStreamSynchronize(J));
    }
    float ms_scan = 0.f, ms_tail = 0.f, ms_all = 0.f, ms_join = 0.f;
    cudaEventElapsedTime(&ms_scan, ev[EV_S0], ev[EV_S1]);
    cudaEventElapsedTime(&ms_all, ev[EV_S0], ev[EV_J1]);
    cudaEventElapsedTime(&ms_join, ev[EV_J0], ev[EV_J1]);
    ms_tail = ms_all - ms_scan;   // what the join adds behind the last block's announcement
    float k1_ms = 0.f;
    for (DetectPending* q : pend) k1_ms += detect_pending_k1_ms(q);

    DevMatchesImpl* impl = new DevMatchesImpl();
    impl->block = fin_owned;
    impl->owner = x->ctx;
    void* fin = fin_owned;
    fin_owned = nullptr;   // the result owns the block now
    out->n_traces = n_tr;
    out->n_occurrences = n_occ;
    out->n_events = n_ev;
    const bool counted = (flags & (SIESTA_F_COUNT_MATCHES | SIESTA_F_RETURN_ALL | SIESTA_F_LITERAL_RUNS)) != 0;
    out->n_matches_emitted = counted ? run.n_emitted : -1;
    out->n_ref_errors = n_err;
    out->kernel_ms = ms_all;
    out->detect_ms = k1_ms;
    out->d_trace_idx = D.trace_idx;
    out->d_occ_off = D.occ_off;
    out->d_ev_off = D.ev_off;
    out->d_ev_pos = D.pos;
    out->d_ev_rank = D.rank;
    out->d_ev_act = D.act;
    out->d_ev_ts_ms = D.ts;
    out->d_err_trace_idx = D.err;
    out->n_unsupported = n_unsup;
    out->d_unsupported_trace_idx = D.unsup;
    out->d_block = fin;
    out->block_bytes = (int64_t)f_bytes;
    out->impl = impl;
    if (stats) {
        int64_t wire = 0;
        for (int b = 0; b < C; ++b)
            for (int p = 0; p < world; ++p) {
                const XHeader& h = hx->hdrs[b * XCHG_MAX_RANKS + p];
                if (p == rank) {
                    stats->local_traces += h.n_tr;
                    stats->local_occurrences += h.n_occ;
                    stats->local_events += h.n_ev;
                    continue;
                }
                wire += h.n_tr * (4 + (all_cols ? 8 : 0)) + (h.uniform_k ? 0 : 4 * (h.n_tr + h.n_occ + 2)) + h.n_ev * (all_cols ? 9 : 2) + 8 * h.n_err;
            }
        stats->k1_ms = k1_ms;
        stats->scan_ms = ms_scan;
        if (C == 1) {   // one block: the phases follow one another
            float ms_wait = 0.f, ms_gap = 0.f, ms_pull = 0.f;
            cudaEventElapsedTime(&ms_wait, ev[EV_S1], ev[EV_H0]);
            cudaEventElapsedTime(&ms_gap, ev[EV_H0], ev[EV_D0]);
            cudaEventElapsedTime(&ms_pull, ev[EV_D0], ev[EV_J1]);
            stats->wait_ms = ms_wait > 0.f ? ms_wait : 0.f;
            stats->host_gap_ms = ms_gap;
            stats->pull_ms = ms_pull;
        } else {
            stats->wait_ms = 0.0;
            stats->pull_ms = ms_tail > 0.f ? ms_tail : 0.f;
            stats->host_gap_ms = 0.0;
        }
        stats->pulled_bytes = wire;
        stats->n_blocks = C;
        stats->eager = eager ? 1 : 0;
        stats->join_ms = ms_join;
    }
    return SIESTA_OK;
}

extern "C" int siesta_exchange_allreduce_i64(siesta_exchange* xh, int64_t* d_buf, int64_t n, int32_t op, void* stream_) {
    Exchange* x = reinterpret_cast<Exchange*>(xh);
    int rc = check_ready(x, "siesta_exchange_allreduce_i64");
    if (rc) return rc;
    if (!d_buf || n < 0 || (op != SIESTA_REDUCE_SUM && op != SIESTA_REDUCE_MIN && op != SIESTA_REDUCE_MAX)) {
        set_error("siesta_exchange_allreduce_i64: bad argument");
        return SIESTA_E_INVALID;
    }
    if ((size_t)n * 8 > x->cap_bytes) {
        set_error("siesta_exchange_allreduce_i64: the array does not fit the exchange region");
        return SIESTA_E_NOMEM;
    }
    std::lock_guard<std::mutex> lock(x->mu);
    SIESTA_CUDA_OK(cudaSetDevice(x->ctx->device));
    cudaStream_t stream = x->stream;
    cudaStream_t user = reinterpret_cast<cudaStream_t>(stream_);
    const unsigned long long seq = ++x->seq;
    XCtrl* me = reinterpret_cast<XCtrl*>(x->region);
    int* d_flag = &x->d_x->flag;
    int* h_flag = &x->h_x->flag;
    // order after the producer of d_buf on the caller's stream
    cudaEvent_t evu;
    SIESTA_CUDA_OK(cudaEventCreateWithFlags(&evu, cudaEventDisableTiming));
    cudaEventRecord(evu, user ? user : x->ctx->stream);
    cudaStreamWaitEvent(stream, evu, 0);
    cudaEventDestroy(evu);
    SIESTA_CUDA_OK(cudaMemsetAsync(d_flag, 0, sizeof(int), stream));
    xchg_wait_acks_kernel<<<1, 32, 0, stream>>>(me, x->world, x->rank, seq - 1, d_flag);
    SIESTA_LAUNCHED();
    XHeader hd;
    std::memset(&hd, 0, sizeof(hd));
    hd.seq = seq;
    SIESTA_CUDA_OK(cudaMemcpyAsync(&me->hdr[0], &hd, sizeof(hd), cudaMemcpyHostToDevice, stream));
    if (n) SIESTA_CUDA_OK(cudaMemcpyAsync(x->region + XCHG_CTRL_BYTES, d_buf, (size_t)n * 8, cudaMemcpyDeviceToDevice, stream));
    xchg_signal_kernel<<<1, 32, 0, stream>>>(x->peers, x->world, x->rank, seq, x->d_x->hdrs, d_flag);
    SIESTA_LAUNCHED();
    if (n) {
        const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)x->ctx->sm_count * 4);
        xchg_reduce_kernel<<<grid, 256, 0, stream>>>(x->peers, x->world, n, op, d_buf);
        SIESTA_LAUNCHED();
    }
    xchg_ack_kernel<<<1, 32, 0, stream>>>(x->peers, x->world, x->rank, seq);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaMemcpyAsync(h_flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    if (*h_flag) {
        set_error("exchange: a peer did not arrive within the time limit");
        return SIESTA_E_CUDA;
    }
    return SIESTA_OK;
}

// ------------------------------------------------------------------------------------------ one process, all GPUs
// The reference is ONE JVM; its drop-in drives every GPU of the box from that process.  siesta_multi owns one context
// and one exchange per device (connected through peer access), siesta_multi_log shards a host CSR log by contiguous
// trace range balanced by event count, and the request entry points run every shard on its own device from its own
// host thread.  /detection results go to the HOST (that is where the JVM needs them), so the shards' match lists are
// joined there: each device copies its columns straight into its slice of one pinned block - eight PCIe links in
// parallel, no device-side all-gather in front of them.  The count arrays are all-reduced on the devices over the
// exchange and read back once.
#include <thread>

namespace siesta {
struct Multi {
    std::vector<Ctx*> ctx;
    std::vector<Exchange*> xchg;
};
struct MultiLog {
    Multi* m = nullptr;
    std::vector<Log*> shard;
    std::vector<int64_t> first;   // first trace of each shard (+ the total at the end)
    int32_t n_activities = 0;
};
}  // namespace siesta

extern "C" int siesta_multi_init(const int32_t* device_ids, int32_t n_dev, siesta_multi** out) {
    if (!device_ids || !out || n_dev < 1 || n_dev > XCHG_MAX_RANKS) {
        set_error("siesta_multi_init: 1..16 device ids");
        return SIESTA_E_INVALID;
    }
    Multi* m = new Multi();
    int rc = SIESTA_OK;
    for (int r = 0; r < n_dev && rc == SIESTA_OK; ++r) {
        siesta_ctx* c = nullptr;
        rc = siesta_init(device_ids[r], &c);
        if (rc == SIESTA_OK) m->ctx.push_back(reinterpret_cast<Ctx*>(c));
    }
    for (int r = 0; r < n_dev && rc == SIESTA_OK; ++r) {
        siesta_exchange* x = nullptr;
        rc = siesta_exchange_create(reinterpret_cast<siesta_ctx*>(m->ctx[r]), n_dev, r, 8 << 20, &x);
        if (rc == SIESTA_OK) m->xchg.push_back(reinterpret_cast<Exchange*>(x));
    }
    for (int a = 0; a < n_dev && rc == SIESTA_OK; ++a)
        for (int b = 0; b < n_dev && rc == SIESTA_OK; ++b)
            if (a != b) rc = siesta_exchange_connect_local(reinterpret_cast<siesta_exchange*>(m->xchg[a]), b, reinterpret_cast<siesta_exchange*>(m->xchg[b]));
    if (rc != SIESTA_OK) {
        const std::string why = siesta_last_error();
        siesta_multi_shutdown(reinterpret_cast<siesta_multi*>(m));
        set_error(why);
        return rc;
    }
    *out = reinterpret_cast<siesta_multi*>(m);
    return SIESTA_OK;
}

extern "C" void siesta_multi_shutdown(siesta_multi* mh) {
    Multi* m = reinterpret_cast<Multi*>(mh);
    if (!m) return;
    for (Exchange* x : m->xchg) siesta_exchange_free(reinterpret_cast<siesta_exchange*>(x));
    for (Ctx* c : m->ctx) siesta_shutdown(reinterpret_cast<siesta_ctx*>(c));
    delete m;
}

extern "C" int32_t siesta_multi_n_devices(const siesta_multi* mh) { return mh ? (int32_t)reinterpret_cast<const Multi*>(mh)->ctx.size() : 0; }

extern "C" int siesta_multi_log_load(siesta_multi* mh, const int64_t* trace_off, const int32_t* act, const int64_t* ts_ms,
                                     int64_t n_traces, int64_t n_events, int32_t n_activities, siesta_multi_log** out) {
    Multi* m = reinterpret_cast<Multi*>(mh);
    if (!m || !trace_off || !out || n_traces < 0 || n_events < 0 || trace_off[0] != 0 || trace_off[n_traces] != n_events) {
        set_error("siesta_multi_log_load: bad argument (trace_off must start at 0 and end at n_events)");
        return SIESTA_E_INVALID;
    }
    const int n = (int)m->ctx.size();
    MultiLog* ml = new MultiLog();
    ml->m = m;
    ml->n_activities = n_activities;
    // contiguous trace ranges balanced by event count (as distributed.shard_bounds)
    ml->first.assign((size_t)n + 1, n_traces);
    ml->first[0] = 0;
    for (int r = 1; r < n; ++r) {
        const int64_t target = (int64_t)((__int128)n_events * r / n);
        const int64_t cut = (int64_t)(std::lower_bound(trace_off, trace_off + n_traces + 1, target) - trace_off);
        ml->first[r] = std::max(ml->first[r - 1], std::min<int64_t>(cut, n_traces));
    }
    int rc = SIESTA_OK;
    std::vector<int64_t> rebased;
    for (int r = 0; r < n && rc == SIESTA_OK; ++r) {
        const int64_t lo = ml->first[r], hi = ml->first[r + 1], e0 = trace_off[lo], e1 = trace_off[hi];
        rebased.assign(trace_off + lo, trace_off + hi + 1);
        for (int64_t& v : rebased) v -= e0;
        siesta_log* lg = nullptr;
        rc = siesta_log_load(reinterpret_cast<siesta_ctx*>(m->ctx[r]), rebased.data(), act ? act + e0 : nullptr, ts_ms ? ts_ms + e0 : nullptr,
                             hi - lo, e1 - e0, n_activities, &lg);
        if (rc == SIESTA_OK) {
            siesta_log_set_first_trace(lg, lo);
            ml->shard.push_back(reinterpret_cast<Log*>(lg));
        }
    }
    if (rc != SIESTA_OK) {
        const std::string why = siesta_last_error();
        siesta_multi_log_free(reinterpret_cast<siesta_multi_log*>(ml));
        set_error(why);
        return rc;
    }
    *out = reinterpret_cast<siesta_multi_log*>(ml);
    return SIESTA_OK;
}

extern "C" void siesta_multi_log_free(siesta_multi_log* lh) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    if (!ml) return;
    for (Log* l : ml->shard) siesta_log_free(reinterpret_cast<siesta_log*>(l));
    delete ml;
}

// The batch is split by shard (new traces go to the last one) with its indices and offsets rebased, and every shard is
// rebuilt by siesta_log_append on its device from its own host thread.  The old multi log is not touched.
extern "C" int siesta_multi_log_append(siesta_multi_log* lh, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                                       const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces, int32_t n_activities,
                                       siesta_multi_log** out) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    if (!ml || !out) {
        set_error("siesta_multi_log_append: null argument");
        return SIESTA_E_INVALID;
    }
    const int n = (int)ml->shard.size();
    const int64_t total = ml->first[(size_t)n];
    if (n_activities < ml->n_activities) {
        set_error("siesta_multi_log_append: n_activities is smaller than the log's (the dictionary only grows)");
        return SIESTA_E_INVALID;
    }
    if (!append_check_batch("siesta_multi_log_append", total, trace_idx, batch_off, n_listed, act, ts_ms, n_new_traces)) return SIESTA_E_INVALID;
    // listed traces [cut[r], cut[r + 1]) belong to shard r
    std::vector<int64_t> cut((size_t)n + 1, n_listed);
    cut[0] = 0;
    for (int r = 1; r < n; ++r) cut[(size_t)r] = (int64_t)(std::lower_bound(trace_idx, trace_idx + n_listed, ml->first[(size_t)r]) - trace_idx);
    std::vector<Log*> built((size_t)n, nullptr);
    std::vector<int> rcs((size_t)n, SIESTA_OK);
    std::vector<std::string> errs((size_t)n);
    {
        std::vector<std::thread> th;
        for (int r = 0; r < n; ++r)
            th.emplace_back([&, r] {
                const int64_t l0 = cut[(size_t)r], l1 = cut[(size_t)r + 1], b0 = batch_off[l0];
                std::vector<int64_t> idx((size_t)(l1 - l0)), off((size_t)(l1 - l0 + 1));
                for (int64_t i = l0; i < l1; ++i) idx[(size_t)(i - l0)] = trace_idx[i] - ml->first[(size_t)r];
                for (int64_t i = l0; i <= l1; ++i) off[(size_t)(i - l0)] = batch_off[i] - b0;
                siesta_log* lg = nullptr;
                rcs[(size_t)r] = siesta_log_append(reinterpret_cast<siesta_log*>(ml->shard[(size_t)r]), idx.data(), off.data(), l1 - l0,
                                                   act ? act + b0 : nullptr, ts_ms ? ts_ms + b0 : nullptr, r == n - 1 ? n_new_traces : 0,
                                                   n_activities, &lg, nullptr);
                if (rcs[(size_t)r] == SIESTA_OK) built[(size_t)r] = reinterpret_cast<Log*>(lg);
                else errs[(size_t)r] = siesta_last_error();
            });
        for (std::thread& t : th) t.join();
    }
    for (int r = 0; r < n; ++r)
        if (rcs[(size_t)r] != SIESTA_OK) {
            for (Log* l : built) siesta_log_free(reinterpret_cast<siesta_log*>(l));
            set_error(errs[(size_t)r]);
            return rcs[(size_t)r];
        }
    MultiLog* nl = new MultiLog();
    nl->m = ml->m;
    nl->shard = built;
    nl->first = ml->first;
    nl->first[(size_t)n] = total + n_new_traces;
    nl->n_activities = n_activities;
    *out = reinterpret_cast<siesta_multi_log*>(nl);
    return SIESTA_OK;
}

extern "C" siesta_log* siesta_multi_log_shard(siesta_multi_log* lh, int32_t r) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    return (ml && r >= 0 && r < (int)ml->shard.size()) ? reinterpret_cast<siesta_log*>(ml->shard[(size_t)r]) : nullptr;
}

// SaseConnector.evaluate + clearOccurrences over the whole (sharded) log: every device verifies its shard at the same
// time; the placements then run in shard order (each needs the sizes of the shards before it to write global offsets)
// and the columns travel to one host block over all host links at once.  Equals siesta_detect on the unsharded log.
extern "C" int siesta_multi_detect(siesta_multi_log* lh, const siesta_nfa* nfa, uint32_t flags, siesta_matches** out) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    if (!ml || !nfa || !out) {
        set_error("siesta_multi_detect: null argument");
        return SIESTA_E_INVALID;
    }
    const int n = (int)ml->shard.size();
    std::vector<DetectPending*> pend((size_t)n, nullptr);
    std::vector<int> rcs((size_t)n, SIESTA_OK);
    std::vector<std::string> errs((size_t)n);
    {   // first halves: all scans in flight
        std::vector<std::thread> th;
        for (int r = 0; r < n; ++r)
            th.emplace_back([&, r] {
                rcs[r] = detect_device_begin_impl(ml->shard[r], nfa, nullptr, 0, flags, ml->shard[r]->ctx->stream, RebaseOffsets{0, 0, 0}, &pend[r]);
                if (rcs[r]) errs[r] = siesta_last_error();
            });
        for (std::thread& t : th) t.join();
    }
    int rc = SIESTA_OK;
    std::vector<siesta_dev_matches> parts((size_t)n);
    for (siesta_dev_matches& p : parts) std::memset(&p, 0, sizeof(p));
    RebaseOffsets base{0, 0, 0};
    for (int r = 0; r < n; ++r) {
        if (rcs[r] != SIESTA_OK) {
            if (rc == SIESTA_OK) {
                rc = rcs[r];
                set_error(errs[r]);
            }
            if (pend[r]) detect_pending_discard(pend[r]);
            continue;
        }
        if (rc != SIESTA_OK) {   // an earlier shard failed: release this one
            siesta_dev_matches tmp;
            detect_device_finish_impl(pend[r], &tmp);
            siesta_dev_matches_free(&tmp);
            continue;
        }
        detect_pending_set_base(pend[r], base);
        rc = detect_device_finish_impl(pend[r], &parts[r]);
        if (rc == SIESTA_OK) {
            base.occ += parts[r].n_occurrences;
            base.ev += parts[r].n_events;
        }
    }
    if (rc == SIESTA_OK) {
        std::vector<Ctx*> pc;
        for (int r = 0; r < n; ++r) pc.push_back(ml->shard[r]->ctx);
        rc = assemble_matches(ml->shard[0]->ctx, parts, flags, nullptr, out, &pc);
        if (rc == SIESTA_OK) {   // device time of a request = the slowest shard, not the sum
            double k = 0, d = 0;
            for (const siesta_dev_matches& p : parts) {
                k = std::max(k, p.kernel_ms);
                d = std::max(d, p.detect_ms);
            }
            (*out)->kernel_ms = k;
            (*out)->detect_ms = d;
        }
    }
    for (siesta_dev_matches& p : parts) siesta_dev_matches_free(&p);
    return rc;
}

// The integer matrices behind /declare over the whole (sharded) log: kernel K3 on every shard, one sum all-reduce over
// the exchange, one read-back.  Equals siesta_declare_counts on the unsharded log.
extern "C" int siesta_multi_declare_counts(siesta_multi_log* lh, int32_t k_cap, int64_t* out, double* kernel_ms) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    if (!ml || !out) {
        set_error("siesta_multi_declare_counts: null argument");
        return SIESTA_E_INVALID;
    }
    const int n = (int)ml->shard.size();
    const int64_t len = siesta_declare_counts_size(ml->n_activities, k_cap);
    if ((size_t)len * 8 > ml->m->xchg[0]->cap_bytes) {
        set_error("siesta_multi_declare_counts: count array larger than the exchange region");
        return SIESTA_E_NOMEM;
    }
    std::vector<int> rcs((size_t)n, SIESTA_OK);
    std::vector<std::string> errs((size_t)n);
    std::vector<double> ms((size_t)n, 0.0);
    std::vector<std::thread> th;
    for (int r = 0; r < n; ++r)
        th.emplace_back([&, r] {
            Ctx* c = ml->shard[r]->ctx;
            int64_t* d = nullptr;
            if (cudaSetDevice(c->device) != cudaSuccess || cudaMallocAsync((void**)&d, (size_t)len * 8, c->stream) != cudaSuccess) {
                rcs[r] = SIESTA_E_NOMEM;
                errs[r] = "siesta_multi_declare_counts: cudaMalloc";
                d = nullptr;
            }
            int rc = rcs[r];
            if (rc == SIESTA_OK) rc = siesta_declare_counts_device(reinterpret_cast<siesta_log*>(ml->shard[r]), k_cap, d, c->stream, &ms[r]);
            // the collective runs even after a local failure (with zeros), so that the other ranks are not left waiting
            if (rc != SIESTA_OK && d) cudaMemsetAsync(d, 0, (size_t)len * 8, c->stream);
            if (rc != SIESTA_OK && errs[r].empty()) errs[r] = siesta_last_error();
            int rc2 = d ? siesta_exchange_allreduce_i64(reinterpret_cast<siesta_exchange*>(ml->m->xchg[r]), d, len, SIESTA_REDUCE_SUM, c->stream) : SIESTA_E_NOMEM;
            if (rc == SIESTA_OK && rc2 != SIESTA_OK) {
                rc = rc2;
                errs[r] = siesta_last_error();
            }
            if (rc == SIESTA_OK && r == 0) {
                if (cudaMemcpyAsync(out, d, (size_t)len * 8, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                    cudaStreamSynchronize(c->stream) != cudaSuccess) {
                    rc = SIESTA_E_CUDA;
                    errs[r] = "siesta_multi_declare_counts: D2H";
                }
            }
            if (d) cudaFreeAsync(d, c->stream);
            rcs[r] = rc;
        });
    for (std::thread& t : th) t.join();
    double worst = 0;
    for (int r = 0; r < n; ++r) {
        worst = std::max(worst, ms[r]);
        if (rcs[r] != SIESTA_OK) {
            set_error(errs[r]);
            return rcs[r];
        }
    }
    if (kernel_ms) *kernel_ms = worst;
    return SIESTA_OK;
}

// siesta_declare_counts_refresh over a sharded log: trace_idx is cut at the shard borders as siesta_multi_log_append cuts
// it (new traces on the last shard); every shard is checked first (no collective runs for a refused call), then every
// shard computes its delta on its device, one sum all-reduce joins the deltas and rank 0 merges them into the old counts.
extern "C" int siesta_multi_declare_counts_refresh(siesta_multi_log* old_h, siesta_multi_log* new_h, const int64_t* trace_idx,
                                                   int64_t n_listed, int32_t k_cap, const int64_t* old_counts, int64_t* out,
                                                   double* kernel_ms) {
    static const char* fn = "siesta_multi_declare_counts_refresh";
    MultiLog* mo = reinterpret_cast<MultiLog*>(old_h);
    MultiLog* mn = reinterpret_cast<MultiLog*>(new_h);
    if (!mo || !mn || !old_counts || !out || n_listed < 0 || (n_listed > 0 && !trace_idx)) {
        set_error(std::string(fn) + ": null argument");
        return SIESTA_E_INVALID;
    }
    const int n = (int)mo->shard.size();
    if (mn->m != mo->m || (int)mn->shard.size() != n) {
        set_error(std::string(fn) + ": the two logs are on different contexts");
        return SIESTA_E_INVALID;
    }
    for (int r = 0; r < n; ++r)
        if (mn->first[(size_t)r] != mo->first[(size_t)r]) {
            set_error(std::string(fn) + ": new_log is not old_log grown by siesta_multi_log_append");
            return SIESTA_E_INVALID;
        }
    const int64_t T = mo->first[(size_t)n], T2 = mn->first[(size_t)n];
    if (T2 < T || mn->n_activities < mo->n_activities) {
        set_error(std::string(fn) + ": new_log has fewer traces or a smaller alphabet than old_log");
        return SIESTA_E_INVALID;
    }
    int64_t n_new = 0;
    for (int64_t i = 0; i < n_listed; ++i) {
        if (trace_idx[i] < 0 || trace_idx[i] >= T2 || (i > 0 && trace_idx[i] <= trace_idx[i - 1])) {
            set_error(std::string(fn) + ": trace_idx must ascend strictly inside [0, new_log's n_traces)");
            return SIESTA_E_INVALID;
        }
        n_new += trace_idx[i] >= T;
    }
    if (n_new != T2 - T) {
        set_error(std::string(fn) + ": trace_idx must list every trace new_log adds (as passed to siesta_multi_log_append)");
        return SIESTA_E_INVALID;
    }
    // listed traces [cut[r], cut[r + 1]) belong to shard r, local indices
    std::vector<int64_t> cut((size_t)n + 1, n_listed);
    cut[0] = 0;
    for (int r = 1; r < n; ++r) cut[(size_t)r] = (int64_t)(std::lower_bound(trace_idx, trace_idx + n_listed, mo->first[(size_t)r]) - trace_idx);
    std::vector<std::vector<int64_t>> idx((size_t)n);
    for (int r = 0; r < n; ++r)
        for (int64_t i = cut[(size_t)r]; i < cut[(size_t)r + 1]; ++i) idx[(size_t)r].push_back(trace_idx[i] - mo->first[(size_t)r]);
    for (int r = 0; r < n; ++r)
        if (!declare_refresh_check_host(fn, mo->shard[(size_t)r], mn->shard[(size_t)r], idx[(size_t)r].data(), (int64_t)idx[(size_t)r].size(), k_cap))
            return SIESTA_E_INVALID;
    const int32_t A0 = mo->n_activities, A1 = mn->n_activities;
    if (A1 < 1 || A1 > 4096) {
        set_error("declare counting: 1 <= n_activities <= 4096 (the eight A x A count matrices of the result)");
        return SIESTA_E_UNSUPPORTED;
    }
    const int64_t len = siesta_declare_counts_size(A1, k_cap), len0 = siesta_declare_counts_size(A0, k_cap);
    if ((size_t)len * 8 > mo->m->xchg[0]->cap_bytes) {
        set_error(std::string(fn) + ": count array larger than the exchange region");
        return SIESTA_E_NOMEM;
    }
    // every shard checks its listed traces on its device before any collective
    std::vector<DeclareRefresh> rr((size_t)n);
    std::vector<int> rcs((size_t)n, SIESTA_OK);
    std::vector<std::string> errs((size_t)n);
    {
        std::vector<std::thread> th;
        for (int r = 0; r < n; ++r)
            th.emplace_back([&, r] {
                DeclareRefresh& x = rr[(size_t)r];
                x.O = mo->shard[(size_t)r];
                x.N = mn->shard[(size_t)r];
                x.n_listed = (int64_t)idx[(size_t)r].size();
                if (cudaSetDevice(x.N->ctx->device) != cudaSuccess) {
                    rcs[(size_t)r] = SIESTA_E_CUDA;
                    errs[(size_t)r] = std::string(fn) + ": cudaSetDevice";
                    return;
                }
                rcs[(size_t)r] = declare_refresh_stage(fn, &x, idx[(size_t)r].data(), x.N->ctx->stream, nullptr);
                if (rcs[(size_t)r]) errs[(size_t)r] = siesta_last_error();
            });
        for (std::thread& t : th) t.join();
    }
    bool full = false;
    for (int r = 0; r < n; ++r) full |= declare_refresh_needs_full(mo->shard[(size_t)r], mn->shard[(size_t)r]);
    auto release_all = [&] {
        for (int r = 0; r < n; ++r) {
            cudaSetDevice(rr[(size_t)r].N->ctx->device);
            declare_refresh_release(&rr[(size_t)r], rr[(size_t)r].N->ctx->stream);
        }
    };
    for (int r = 0; r < n; ++r)
        if (rcs[(size_t)r] != SIESTA_OK) {
            release_all();
            set_error(errs[(size_t)r]);
            return rcs[(size_t)r];
        }
    if (full) {   // ids outside the old alphabet that the new one covers: count the new log in full (the header's fallback)
        release_all();
        return siesta_multi_declare_counts(new_h, k_cap, out, kernel_ms);
    }
    std::vector<double> ms((size_t)n, 0.0);
    std::vector<std::thread> th;
    for (int r = 0; r < n; ++r)
        th.emplace_back([&, r] {
            DeclareRefresh& x = rr[(size_t)r];
            Ctx* c = x.N->ctx;
            cudaSetDevice(c->device);
            int64_t* d = nullptr;
            int64_t* d_old = nullptr;
            cudaEvent_t e0 = nullptr, e1 = nullptr;
            int rc = SIESTA_OK;
            if (cudaMallocAsync((void**)&d, (size_t)len * 8, c->stream) != cudaSuccess) {
                rc = SIESTA_E_NOMEM;
                errs[(size_t)r] = std::string(fn) + ": cudaMalloc";
                d = nullptr;
            }
            if (rc == SIESTA_OK && (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess ||
                                    cudaEventRecord(e0, c->stream) != cudaSuccess)) {
                rc = SIESTA_E_CUDA;
                errs[(size_t)r] = std::string(fn) + ": cudaEvent";
            }
            if (rc == SIESTA_OK) rc = declare_refresh_delta(&x, k_cap, d, c->stream);
            // the collective runs even after a local failure (with zeros), so that the other ranks are not left waiting
            if (rc != SIESTA_OK && d) cudaMemsetAsync(d, 0, (size_t)len * 8, c->stream);
            if (rc != SIESTA_OK && errs[(size_t)r].empty()) errs[(size_t)r] = siesta_last_error();
            int rc2 = d ? siesta_exchange_allreduce_i64(reinterpret_cast<siesta_exchange*>(mo->m->xchg[(size_t)r]), d, len, SIESTA_REDUCE_SUM, c->stream)
                        : SIESTA_E_NOMEM;
            if (rc == SIESTA_OK && rc2 != SIESTA_OK) {
                rc = rc2;
                errs[(size_t)r] = siesta_last_error();
            }
            if (rc == SIESTA_OK && r == 0) {
                if (cudaMallocAsync((void**)&d_old, (size_t)len0 * 8, c->stream) != cudaSuccess ||
                    cudaMemcpyAsync(d_old, old_counts, (size_t)len0 * 8, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
                    rc = SIESTA_E_CUDA;
                    errs[(size_t)r] = std::string(fn) + ": H2D of the old counts";
                }
                if (rc == SIESTA_OK) rc = declare_merge(d_old, A0, A1, k_cap, d, d, c, c->stream);
                if (rc != SIESTA_OK && errs[(size_t)r].empty()) errs[(size_t)r] = siesta_last_error();
                if (rc == SIESTA_OK && cudaEventRecord(e1, c->stream) != cudaSuccess) rc = SIESTA_E_CUDA;
                if (rc == SIESTA_OK && (cudaMemcpyAsync(out, d, (size_t)len * 8, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                                        cudaStreamSynchronize(c->stream) != cudaSuccess)) {
                    rc = SIESTA_E_CUDA;
                    errs[(size_t)r] = std::string(fn) + ": D2H";
                }
            } else if (rc == SIESTA_OK && cudaEventRecord(e1, c->stream) != cudaSuccess) {
                rc = SIESTA_E_CUDA;
            }
            float f = 0.f;
            if (rc == SIESTA_OK && cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&f, e0, e1) == cudaSuccess) ms[(size_t)r] = f;
            if (d_old) cudaFreeAsync(d_old, c->stream);
            if (d) cudaFreeAsync(d, c->stream);
            declare_refresh_release(&x, c->stream);
            if (e0) cudaEventDestroy(e0);
            if (e1) cudaEventDestroy(e1);
            rcs[(size_t)r] = rc;
        });
    for (std::thread& t : th) t.join();
    double worst = 0;
    for (int r = 0; r < n; ++r) {
        worst = std::max(worst, ms[(size_t)r]);
        if (rcs[(size_t)r] != SIESTA_OK) {
            set_error(errs[(size_t)r]);
            return rcs[(size_t)r];
        }
    }
    if (kernel_ms) *kernel_ms = worst;
    return SIESTA_OK;
}


// Why-not-match over a sharded log: the candidates (global trace indices, ascending) are cut at the shard borders, every
// device evaluates its own (siesta_why_not_match on the shard, wnm.cu), the answers are concatenated in shard order -
// traces are independent, nothing crosses a device.
extern "C" int siesta_multi_why_not_match(siesta_multi_log* lh, const int32_t* pattern, int32_t m, const siesta_wnm_constraint* cons,
                                          int32_t n_cons, int32_t uncertainty, int32_t step, int32_t k, const int64_t* cand,
                                          int64_t n_cand, uint32_t flags, siesta_almost_matches** out) {
    MultiLog* ml = reinterpret_cast<MultiLog*>(lh);
    if (!ml || !out || (cand == nullptr && n_cand != 0) || n_cand < 0) {
        set_error("siesta_multi_why_not_match: null argument");
        return SIESTA_E_INVALID;
    }
    const int n = (int)ml->shard.size();
    for (int64_t i = 0; i < n_cand; ++i)
        if (cand[i] < 0 || cand[i] >= ml->first[(size_t)n] || (i && cand[i] < cand[i - 1])) {
            set_error("siesta_multi_why_not_match: candidates must be ascending trace indices of the log");
            return SIESTA_E_INVALID;
        }
    std::vector<siesta_almost_matches*> part((size_t)n, nullptr);
    std::vector<int> rcs((size_t)n, SIESTA_OK);
    std::vector<std::string> errs((size_t)n);
    std::vector<std::thread> th;
    for (int r = 0; r < n; ++r)
        th.emplace_back([&, r] {
            std::vector<int64_t> local;
            const int64_t* lp = nullptr;
            int64_t ln = 0;
            if (cand) {
                const int64_t* a = std::lower_bound(cand, cand + n_cand, ml->first[(size_t)r]);
                const int64_t* b = std::lower_bound(cand, cand + n_cand, ml->first[(size_t)r + 1]);
                local.assign(a, b);
                for (int64_t& t : local) t -= ml->first[(size_t)r];
                local.push_back(0);   // never a null pointer: null means "every trace"
                lp = local.data();
                ln = (int64_t)local.size() - 1;
            }
            rcs[r] = siesta_why_not_match(reinterpret_cast<siesta_log*>(ml->shard[r]), pattern, m, cons, n_cons, uncertainty, step, k, lp, ln,
                                          flags, &part[r]);
            if (rcs[r]) errs[r] = siesta_last_error();
        });
    for (std::thread& t : th) t.join();
    int rc = SIESTA_OK;
    int64_t n_hit = 0, n_unsup = 0;
    double ms = 0;
    for (int r = 0; r < n; ++r) {
        if (rcs[r] != SIESTA_OK && rc == SIESTA_OK) {
            rc = rcs[r];
            set_error(errs[r]);
        }
        if (part[r]) {
            n_hit += part[r]->n_traces;
            n_unsup += part[r]->n_unsupported;
            ms = std::max(ms, part[r]->kernel_ms);
        }
    }
    siesta_almost_matches* res = nullptr;
    if (rc == SIESTA_OK) {
        const size_t h = (size_t)std::max<int64_t>(n_hit, 1), ev = h * (size_t)m, us = (size_t)std::max<int64_t>(n_unsup, 1);
        char* base = (char*)std::malloc(((sizeof(siesta_almost_matches) + 63) & ~(size_t)63) + h * 12 + us * 8 + ev * 16 + 64);
        if (!base) rc = SIESTA_E_NOMEM;
        else {
            res = reinterpret_cast<siesta_almost_matches*>(base);
            std::memset(res, 0, sizeof(*res));
            char* p = base + ((sizeof(siesta_almost_matches) + 63) & ~(size_t)63);
            res->trace_idx = reinterpret_cast<int64_t*>(p); p += h * 8;
            res->unsupported_trace_idx = reinterpret_cast<int64_t*>(p); p += us * 8;
            res->total_change = reinterpret_cast<int32_t*>(p); p += h * 4;
            res->ev_pos = reinterpret_cast<int32_t*>(p); p += ev * 4;
            res->ev_value = reinterpret_cast<int32_t*>(p); p += ev * 4;
            res->ev_change = reinterpret_cast<int32_t*>(p); p += ev * 4;
            res->ev_stream_pos = reinterpret_cast<int32_t*>(p);
            res->n_states = m;
            res->kernel_ms = ms;
            for (int r = 0; r < n; ++r) {
                const siesta_almost_matches* q = part[r];
                std::memcpy(res->trace_idx + res->n_traces, q->trace_idx, (size_t)q->n_traces * 8);
                std::memcpy(res->total_change + res->n_traces, q->total_change, (size_t)q->n_traces * 4);
                std::memcpy(res->ev_pos + res->n_traces * m, q->ev_pos, (size_t)q->n_traces * m * 4);
                std::memcpy(res->ev_value + res->n_traces * m, q->ev_value, (size_t)q->n_traces * m * 4);
                std::memcpy(res->ev_change + res->n_traces * m, q->ev_change, (size_t)q->n_traces * m * 4);
                std::memcpy(res->ev_stream_pos + res->n_traces * m, q->ev_stream_pos, (size_t)q->n_traces * m * 4);
                std::memcpy(res->unsupported_trace_idx + res->n_unsupported, q->unsupported_trace_idx, (size_t)q->n_unsupported * 8);
                res->n_traces += q->n_traces;
                res->n_unsupported += q->n_unsupported;
            }
        }
    }
    for (siesta_almost_matches* q : part) siesta_almost_matches_free(q);
    if (rc != SIESTA_OK) return rc;
    *out = res;
    return SIESTA_OK;
}
