// declare.cu — kernel K3: per-trace counting behind /declare (existences, ordered relations, positions).
//
// Replaces the Spark jobs of QueryPlanExistences (createMapForSingle :136-142, joinUnionTraces :164-179),
// QueryPlanOrderedRelations (joinTables :97-116, evaluateConstraint :127-151 with
// OrderedRelationsUtilityFunctions.countResponse/countPrecedence :25-44) and QueryPlanPositions.execute :51-79
// (all under J/declare/queryPlans/).  The kernel produces integer count matrices; supports (one double division)
// and thresholds stay on the host, fed by these integers.
//
// One warp per trace.  Pass 1 (lanes = events, coalesced int32 loads): per-activity count / first / last position
// in the warp's shared-memory scratch.  Pass 2 (lanes = activities): existence histogram and the A x A presence
// matrices from (count, first, last) alone.  Pass 3 (serial over the trace, lanes = activities): response and
// precedence through running per-activity counts, touched only at the first / last occurrence of an activity:
//     response[a][b]   = #{a : some b after a}  = (# a before last[b])
//     precedence[a][b] = #{b : some a before b} = count[b] - (# b before first[a])
// All counters of a CTA live in shared memory (uint32) and are flushed with 64-bit atomics once per CTA.
// Bound: integer ALU / shared-memory atomics, not HBM (4 B/event + 8 B/trace of traffic); see DESIGN.md.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace siesta {

constexpr int DT = 256;      // threads per CTA
constexpr int DTS_MAX = 1024;   // the serial kernels: CTA size chosen per launch (shared-memory matrices are per CTA: large alphabets
                                // fit one CTA per SM, which then has to hold all the SM's warps)
constexpr int HS = 16;       // histogram buckets kept in shared memory (k < HS)
constexpr int MAX_A_SMEM = 104;   // the serial kernels keep four A x A matrices in shared memory
constexpr int MAX_A_ANY = 4096;   // declare_any_kernel: bounded by the result itself (8 A^2 int64 = 1 GB)

struct DeclareParams {
    const int64_t* trace_off;
    const int32_t* act;
    int64_t n_traces;         // rows of the launch: the log's traces, or the entries of `work`
    int32_t A;
    int32_t k_cap;
    unsigned long long* out;  // packed layout, see siesta_declare_counts_size
    const int64_t* work;      // work-list launches (WL): row i is trace work[i]
    int32_t neg;              // work-list launches: 1 = subtract the rows' counts from `out` (wrapping 64-bit arithmetic)
};

// Work-list mode (the count refresh after a log append): the kernels take a template flag WL.  With WL, row i of the
// launch is trace P.work[i] and every count that reaches the result passes sgn() (negated when P.neg).  Without it both
// helpers are the identity, so the full-log instantiations compile to the code they had before the mode existed.
template <bool WL>
__device__ __forceinline__ long long row_trace(const DeclareParams& P, long long i) {
    if constexpr (WL) return P.work[i];
    else return i;
}
template <bool WL>
__device__ __forceinline__ unsigned long long sgn(const DeclareParams& P, unsigned long long v) {
    if constexpr (WL) return P.neg ? 0ull - v : v;
    else return v;
}

__device__ __forceinline__ long long shfl64(long long v, int src) {
    int lo = __shfl_sync(0xffffffffu, (int)(v & 0xffffffffll), src);
    int hi = __shfl_sync(0xffffffffu, (int)(v >> 32), src);
    return ((long long)hi << 32) | (unsigned int)lo;
}

template <int NB, bool WL>  // NB = ceil(A / 32) activity blocks held in registers per lane
__global__ void __launch_bounds__(DTS_MAX) declare_kernel(const __grid_constant__ DeclareParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int A = P.A;
    const int AA = A * A;
    uint32_t* s_co = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* s_ord = s_co + AA;
    uint32_t* s_respT = s_ord + AA;   // transposed: [b][a]
    uint32_t* s_prec = s_respT + AA;  // [a][b]
    uint32_t* s_tot = s_prec + AA;
    uint32_t* s_uniq = s_tot + A;
    uint32_t* s_first = s_uniq + A;
    uint32_t* s_last = s_first + A;
    uint32_t* s_hist = s_last + A;    // [A][HS]
    uint32_t* s_warp = s_hist + A * HS;  // per warp: cnt[A], first[A], last[A]
    __shared__ unsigned long long s_misc[2];  // hist_overflow, n_nonempty

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* w_cnt = s_warp + warp * 3 * A;
    uint32_t* w_first = w_cnt + A;
    uint32_t* w_last = w_first + A;

    for (int i = threadIdx.x; i < 4 * AA + 4 * A + A * HS; i += blockDim.x) s_co[i] = 0;
    if (threadIdx.x < 2) s_misc[threadIdx.x] = 0;
    __syncthreads();

    const long long warps_total = (long long)gridDim.x * (blockDim.x / 32);
    for (long long t = (long long)blockIdx.x * (blockDim.x / 32) + warp; t < P.n_traces; t += warps_total) {
        long long lo = 0, hi = 0;
        if (lane == 0) { const long long tr = row_trace<WL>(P, t); lo = P.trace_off[tr]; hi = P.trace_off[tr + 1]; }
        lo = shfl64(lo, 0);
        hi = shfl64(hi, 0);
        if (hi <= lo) continue;
        const int len = (int)(hi - lo);
        for (int a = lane; a < A; a += 32) { w_cnt[a] = 0; w_first[a] = 0xffffffffu; w_last[a] = 0; }
        __syncwarp();
        // pass 1: per-activity count / first / last
        for (int i = lane; i < len; i += 32) {
            const int x = __ldg(P.act + lo + i);
            if (x >= 0 && x < A) {
                atomicAdd(&w_cnt[x], 1u);
                atomicMin(&w_first[x], (uint32_t)i);
                atomicMax(&w_last[x], (uint32_t)i);
            }
        }
        __syncwarp();
        if (lane == 0) {
            atomicAdd(&s_misc[1], 1ull);
            const int xf = P.act[lo], xl = P.act[hi - 1];
            if (xf >= 0 && xf < A) atomicAdd(&s_first[xf], 1u);
            if (xl >= 0 && xl < A) atomicAdd(&s_last[xl], 1u);
        }
        // pass 2: existence counts and presence matrices
        uint32_t cnt_r[NB], run_r[NB];
#pragma unroll
        for (int kb = 0; kb < NB; ++kb) {
            const int b = kb * 32 + lane;
            cnt_r[kb] = b < A ? w_cnt[b] : 0;
            run_r[kb] = 0;
            if (cnt_r[kb]) {
                atomicAdd(&s_tot[b], cnt_r[kb]);
                atomicAdd(&s_uniq[b], 1u);
                if (cnt_r[kb] > (uint32_t)P.k_cap) atomicAdd(&s_misc[0], 1ull);   // beyond the caller's histogram
                else if (cnt_r[kb] < (uint32_t)HS) atomicAdd(&s_hist[b * HS + cnt_r[kb]], 1u);
                else atomicAdd(P.out + 4ll * A + (long long)b * (P.k_cap + 1) + cnt_r[kb], sgn<WL>(P, 1ull));
            }
        }
        for (int a = 0; a < A; ++a) {
            const uint32_t ca = w_cnt[a];
            if (ca == 0) continue;  // uniform
            const uint32_t fa = w_first[a];
#pragma unroll
            for (int kb = 0; kb < NB; ++kb) {
                const int b = kb * 32 + lane;
                if (b >= A || cnt_r[kb] == 0) continue;
                if (b == a) {
                    if (ca >= 2) { atomicAdd(&s_ord[a * A + b], 1u); atomicAdd(&s_co[a * A + b], 1u); }
                } else {
                    atomicAdd(&s_co[a * A + b], 1u);
                    if (fa < w_last[b]) atomicAdd(&s_ord[a * A + b], 1u);
                }
            }
        }
        // pass 3: response / precedence at first / last occurrences, running counts in registers
        for (int i = 0; i < len; ++i) {
            const int x = __ldg(P.act + lo + i);  // uniform address: one broadcast transaction
            if (x < 0 || x >= A) continue;
            const bool is_last = w_last[x] == (uint32_t)i, is_first = w_first[x] == (uint32_t)i;
            if (is_last || is_first) {
#pragma unroll
                for (int kb = 0; kb < NB; ++kb) {
                    const int o = kb * 32 + lane;
                    if (o >= A || o == x || cnt_r[kb] == 0) continue;
                    if (is_last && run_r[kb]) atomicAdd(&s_respT[x * A + o], run_r[kb]);               // response[o][x]
                    if (is_first && cnt_r[kb] > run_r[kb]) atomicAdd(&s_prec[x * A + o], cnt_r[kb] - run_r[kb]);  // precedence[x][o]
                }
            }
#pragma unroll
            for (int kb = 0; kb < NB; ++kb)
                if (x == kb * 32 + lane) ++run_r[kb];
        }
        __syncwarp();
    }
    __syncthreads();
    // flush: packed layout tot uniq first last hist co ordered response precedence overflow nonempty
    unsigned long long* o_tot = P.out;
    unsigned long long* o_uniq = o_tot + A;
    unsigned long long* o_first = o_uniq + A;
    unsigned long long* o_last = o_first + A;
    unsigned long long* o_hist = o_last + A;
    unsigned long long* o_co = o_hist + (long long)A * (P.k_cap + 1);
    unsigned long long* o_ord = o_co + AA;
    unsigned long long* o_resp = o_ord + AA;
    unsigned long long* o_prec = o_resp + AA;
    for (int i = threadIdx.x; i < A; i += blockDim.x) {
        if (s_tot[i]) atomicAdd(o_tot + i, sgn<WL>(P, s_tot[i]));
        if (s_uniq[i]) atomicAdd(o_uniq + i, sgn<WL>(P, s_uniq[i]));
        if (s_first[i]) atomicAdd(o_first + i, sgn<WL>(P, s_first[i]));
        if (s_last[i]) atomicAdd(o_last + i, sgn<WL>(P, s_last[i]));
    }
    for (int i = threadIdx.x; i < A * HS; i += blockDim.x) {
        const int a = i / HS, k = i % HS;
        if (s_hist[i] && k <= P.k_cap) atomicAdd(o_hist + (long long)a * (P.k_cap + 1) + k, sgn<WL>(P, s_hist[i]));
    }
    for (int i = threadIdx.x; i < AA; i += blockDim.x) {
        if (s_co[i]) atomicAdd(o_co + i, sgn<WL>(P, s_co[i]));
        if (s_ord[i]) atomicAdd(o_ord + i, sgn<WL>(P, s_ord[i]));
        if (s_prec[i]) atomicAdd(o_prec + i, sgn<WL>(P, s_prec[i]));
        if (s_respT[i]) {
            const int b = i / A, a = i % A;  // transposed in shared memory
            atomicAdd(o_resp + (long long)a * A + b, sgn<WL>(P, s_respT[i]));
        }
    }
    if (threadIdx.x == 0) {
        if (s_misc[0]) atomicAdd(o_prec + 5ll * AA, sgn<WL>(P, s_misc[0]));
        if (s_misc[1]) atomicAdd(o_prec + 5ll * AA + 1, sgn<WL>(P, s_misc[1]));
    }
}

// Alternate and chain modes of the ordered relations (OrderedRelationsUtilityFunctions.java:51-102).  Per trace listed
// under (a,b), a != b:
//   countResponseAlternate   = #{ i : some b strictly between a_i and a_(i+1) } + [some b after the last a]
//   countPrecedenceAlternate = #{ i : some a strictly between b_(i-1) and b_i } + [some a before the first b]
// Both count the b's whose nearest earlier event among {a, b} is an a, so they are equal; likewise
//   countResponseChain = #{a : b at position a + 1} = #{b : a at position b - 1} = countPrecedenceChain.
// (tests/test_counting_oracle.py checks the four literal restatements of the oracle against each other.)
// One warp per trace, serial over the events, lanes = activities: lane o keeps the last position of activity o; at an
// event of activity x every lane whose last position is later than x's previous one adds 1 to alternate[o][x].
template <int NB, bool WL>
__global__ void __launch_bounds__(DTS_MAX) declare_alt_chain_kernel(const __grid_constant__ DeclareParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int A = P.A;
    const int AA = A * A;
    uint32_t* s_altT = reinterpret_cast<uint32_t*>(smem_raw);  // transposed: [x][o] = alternate[o][x]
    uint32_t* s_chain = s_altT + AA;                           // [a][b]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 2 * AA; i += blockDim.x) s_altT[i] = 0;
    __syncthreads();
    const long long warps_total = (long long)gridDim.x * (blockDim.x / 32);
    for (long long t = (long long)blockIdx.x * (blockDim.x / 32) + warp; t < P.n_traces; t += warps_total) {
        long long lo = 0, hi = 0;
        if (lane == 0) { const long long tr = row_trace<WL>(P, t); lo = P.trace_off[tr]; hi = P.trace_off[tr + 1]; }
        lo = shfl64(lo, 0);
        hi = shfl64(hi, 0);
        const int len = (int)(hi - lo);
        int last_r[NB];
#pragma unroll
        for (int kb = 0; kb < NB; ++kb) last_r[kb] = -1;
        int px = -1;  // activity of the previous event
        for (int base = 0; base < len; base += 32) {
            const int mine = base + lane < len ? __ldg(P.act + lo + base + lane) : -1;  // 32 events per coalesced load
            const int n_here = len - base < 32 ? len - base : 32;
            for (int k = 0; k < n_here; ++k) {
                const int x = __shfl_sync(0xffffffffu, mine, k);
                const int i = base + k;
                if (x < 0 || x >= A) { px = -1; continue; }
                int prev = -1;  // previous position of x: register (x >> 5) of lane (x & 31)
#pragma unroll
                for (int kb = 0; kb < NB; ++kb)
                    if ((x >> 5) == kb) prev = __shfl_sync(0xffffffffu, last_r[kb], x & 31);
#pragma unroll
                for (int kb = 0; kb < NB; ++kb) {
                    const int o = kb * 32 + lane;
                    if (o < A && o != x && last_r[kb] > prev) atomicAdd(&s_altT[x * A + o], 1u);
                    if (o == x) last_r[kb] = i;
                }
                if (lane == 0 && px >= 0 && px != x) atomicAdd(&s_chain[px * A + x], 1u);
                px = x;
            }
        }
    }
    __syncthreads();
    unsigned long long* o_alt_r = P.out + 4ll * A + (long long)A * (P.k_cap + 1) + 4ll * AA;
    unsigned long long* o_alt_p = o_alt_r + AA;
    unsigned long long* o_chain_r = o_alt_p + AA;
    unsigned long long* o_chain_p = o_chain_r + AA;
    for (int i = threadIdx.x; i < AA; i += blockDim.x) {
        if (s_altT[i]) {
            const int x = i / A, o = i % A;
            atomicAdd(o_alt_r + (long long)o * A + x, sgn<WL>(P, s_altT[i]));
            atomicAdd(o_alt_p + (long long)o * A + x, sgn<WL>(P, s_altT[i]));
        }
        if (s_chain[i]) {
            atomicAdd(o_chain_r + i, sgn<WL>(P, s_chain[i]));
            atomicAdd(o_chain_p + i, sgn<WL>(P, s_chain[i]));
        }
    }
}


// ---------------------------------------------------------------------------------- K3 v2: position masks + pair-owned counters
// For alphabets of at most 32 activities and traces of at most 32 * NW <= 128 events every count of a trace follows from the
// per-activity POSITION MASKS M[a] (bit i <=> event i is an a), with BL[b] = bits below the last b and AF[a] = bits
// above the first a:
//     response[a][b]   += popc(M[a] & BL[b])              #{a : some b after a}   (countResponse :25-31)
//     precedence[a][b] += popc(M[b] & AF[a])              #{b : some a before b}  (countPrecedence :38-44)
//     ordered[a][b]    += (M[a] & BL[b]) != 0             first a < last b        (queryIndexTableDeclare :389-404)
//     co[a][b]         += ordered(a,b) or ordered(b,a)    both present, a != b    (joinUnionTraces :164-179)
//     alternate[a][b]  += popc((~M[b] + M[a]) & M[b])     the b's whose nearest earlier event among {a, b} is an a: adding
//                         M[a] to ~M[b] lets a carry run from every a through the slots that hold no b and land on the next
//                         b (countResponseAlternate :51-60 = countPrecedenceAlternate :67-76, see declare_alt_chain_kernel)
// A CTA works on batches of TB traces.  Phase 1, one warp per trace, lanes = events: __match_any_sync groups the 32
// events of a chunk by activity and the group's leader stores the group mask as one word of M[activity] (shared memory);
// then lanes = activities derive BL / AF, the existence counts (tot, uniq, hist, diagonal) and lanes = events count the
// chain pairs.  Phase 2, one THREAD per unordered activity pair {a < b}: it reads the six masks of its pair for each of
// the TB traces and keeps the nine counters of the pair in registers for the whole launch: no atomics, no serial pass
// over the events.  Cost per trace: ~70 warp instructions (phase 1) + 54 per pair-thread warp (phase 2), against ~2 000
// of the serial kernels above.  Longer traces or larger alphabets keep those kernels.
constexpr int TB = 32;  // traces per batch

// Position mask of NW 32-bit words (2: traces <= 64 events, 3: <= 96, 4: <= 128); 3 words are stored padded to 16 bytes.
template <int NW>
struct PosMask {
    static constexpr int STORE = NW == 3 ? 4 : NW;
    struct alignas(NW == 2 ? 8 : 16) T { uint32_t w[STORE]; };
    static __device__ __forceinline__ T zero() {
        T r;
#pragma unroll
        for (int i = 0; i < STORE; ++i) r.w[i] = 0;
        return r;
    }
    static __device__ __forceinline__ int popc(const T& m) {
        int n = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) n += __popc(m.w[i]);
        return n;
    }
    static __device__ __forceinline__ int popc_and(const T& a, const T& b) {
        int n = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) n += __popc(a.w[i] & b.w[i]);
        return n;
    }
    // bits below the highest set bit (0 for an empty mask)
    static __device__ __forceinline__ T below_last(const T& m) {
        T r = zero();
        bool found = false;
#pragma unroll
        for (int i = NW - 1; i >= 0; --i) {
            if (found) r.w[i] = ~0u;
            else if (m.w[i]) { r.w[i] = ~(~0u << (31 - __clz(m.w[i]))); found = true; }
        }
        return r;
    }
    // bits above the lowest set bit (0 for an empty mask)
    static __device__ __forceinline__ T above_first(const T& m) {
        T r = zero();
        bool found = false;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            if (found) r.w[i] = ~0u;
            else if (m.w[i]) { const uint32_t b = m.w[i] & (0u - m.w[i]); r.w[i] = ~(b | (b - 1u)); found = true; }
        }
        return r;
    }
    // popc((~mb + ma) & mb): one carry chain over the NW words
    static __device__ __forceinline__ int alt(const T& ma, const T& mb) {
        uint32_t s[NW];
        // one asm statement per chain: the carry flag is not visible to the compiler
        if constexpr (NW == 2)
            asm("add.cc.u32 %0, %2, %4;\n\taddc.u32 %1, %3, %5;"
                : "=r"(s[0]), "=r"(s[1]) : "r"(~mb.w[0]), "r"(~mb.w[1]), "r"(ma.w[0]), "r"(ma.w[1]));
        else if constexpr (NW == 3)
            asm("add.cc.u32 %0, %3, %6;\n\taddc.cc.u32 %1, %4, %7;\n\taddc.u32 %2, %5, %8;"
                : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]) : "r"(~mb.w[0]), "r"(~mb.w[1]), "r"(~mb.w[2]), "r"(ma.w[0]), "r"(ma.w[1]), "r"(ma.w[2]));
        else
            asm("add.cc.u32 %0, %4, %8;\n\taddc.cc.u32 %1, %5, %9;\n\taddc.cc.u32 %2, %6, %10;\n\taddc.u32 %3, %7, %11;"
                : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3])
                : "r"(~mb.w[0]), "r"(~mb.w[1]), "r"(~mb.w[2]), "r"(~mb.w[3]), "r"(ma.w[0]), "r"(ma.w[1]), "r"(ma.w[2]), "r"(ma.w[3]));
        int n = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) n += __popc(s[i] & mb.w[i]);
        return n;
    }
};

// NW = 32-bit words per mask; PPT = activity pairs per thread
template <int NW, int PPT, bool WL>
__global__ void __launch_bounds__(256, 3) declare_pairs_kernel(const __grid_constant__ DeclareParams P) {
    typedef PosMask<NW> PM;
    typedef typename PM::T mask_t;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int A = P.A, AA = A * A;
    mask_t* sM = reinterpret_cast<mask_t*>(smem_raw);   // [TB][A]
    mask_t* sBL = sM + TB * A;
    mask_t* sAF = sBL + TB * A;
    uint32_t* s_chain = reinterpret_cast<uint32_t*>(sAF + TB * A);  // [A][A]
    uint32_t* s_first = s_chain + AA;
    uint32_t* s_last = s_first + A;
    uint32_t* s_hist = s_last + A;                                   // [A][HS]
    __shared__ unsigned long long s_misc[2];                         // hist_overflow, n_nonempty

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    for (int i = threadIdx.x; i < AA + 2 * A + A * HS; i += blockDim.x) s_chain[i] = 0;
    if (threadIdx.x < 2) s_misc[threadIdx.x] = 0;

    // the pairs {a < b} of this thread: pair index q = threadIdx.x + j * blockDim.x, row-major over a
    int pa[PPT], pb[PPT];
    const int n_pairs = A * (A - 1) / 2;
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
        int q = threadIdx.x + j * blockDim.x;
        pa[j] = pb[j] = -1;
        if (q < n_pairs) {
            int a = 0;
            while (q >= A - 1 - a) { q -= A - 1 - a; ++a; }
            pa[j] = a;
            pb[j] = a + 1 + q;
        }
    }
    uint32_t c_co[PPT], c_ord_ab[PPT], c_ord_ba[PPT], c_r_ab[PPT], c_r_ba[PPT], c_p_ab[PPT], c_p_ba[PPT], c_alt_ab[PPT], c_alt_ba[PPT];
#pragma unroll
    for (int j = 0; j < PPT; ++j) c_co[j] = c_ord_ab[j] = c_ord_ba[j] = c_r_ab[j] = c_r_ba[j] = c_p_ab[j] = c_p_ba[j] = c_alt_ab[j] = c_alt_ba[j] = 0;
    // lanes = activities (phase 1): existence counts of activity `lane`, summed over the traces this warp builds
    unsigned long long a_tot = 0, a_uniq = 0, a_diag = 0, w_nonempty = 0, w_hist_ovf = 0;
    __syncthreads();

    unsigned long long* o_tot = P.out;
    unsigned long long* o_uniq = o_tot + A;
    unsigned long long* o_first = o_uniq + A;
    unsigned long long* o_last = o_first + A;
    unsigned long long* o_hist = o_last + A;
    unsigned long long* o_co = o_hist + (long long)A * (P.k_cap + 1);
    unsigned long long* o_ord = o_co + AA;
    unsigned long long* o_resp = o_ord + AA;
    unsigned long long* o_prec = o_resp + AA;
    unsigned long long* o_alt_r = o_prec + AA;
    unsigned long long* o_alt_p = o_alt_r + AA;
    unsigned long long* o_chain_r = o_alt_p + AA;
    unsigned long long* o_chain_p = o_chain_r + AA;

    auto flush_pairs = [&]() {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (pa[j] < 0) continue;
            const long long ab = (long long)pa[j] * A + pb[j], ba = (long long)pb[j] * A + pa[j];
            if (c_co[j]) { atomicAdd(o_co + ab, sgn<WL>(P, c_co[j])); atomicAdd(o_co + ba, sgn<WL>(P, c_co[j])); }
            if (c_ord_ab[j]) atomicAdd(o_ord + ab, sgn<WL>(P, c_ord_ab[j]));
            if (c_ord_ba[j]) atomicAdd(o_ord + ba, sgn<WL>(P, c_ord_ba[j]));
            if (c_r_ab[j]) atomicAdd(o_resp + ab, sgn<WL>(P, c_r_ab[j]));
            if (c_r_ba[j]) atomicAdd(o_resp + ba, sgn<WL>(P, c_r_ba[j]));
            if (c_p_ab[j]) atomicAdd(o_prec + ab, sgn<WL>(P, c_p_ab[j]));
            if (c_p_ba[j]) atomicAdd(o_prec + ba, sgn<WL>(P, c_p_ba[j]));
            if (c_alt_ab[j]) { atomicAdd(o_alt_r + ab, sgn<WL>(P, c_alt_ab[j])); atomicAdd(o_alt_p + ab, sgn<WL>(P, c_alt_ab[j])); }
            if (c_alt_ba[j]) { atomicAdd(o_alt_r + ba, sgn<WL>(P, c_alt_ba[j])); atomicAdd(o_alt_p + ba, sgn<WL>(P, c_alt_ba[j])); }
            c_co[j] = c_ord_ab[j] = c_ord_ba[j] = c_r_ab[j] = c_r_ba[j] = c_p_ab[j] = c_p_ba[j] = c_alt_ab[j] = c_alt_ba[j] = 0;
        }
    };

    const long long n_batches = (P.n_traces + TB - 1) / TB;
    int since_flush = 0;
    for (long long batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
        // ---------------------------------------------------------------- phase 1: masks of the batch's traces
        for (int slot = warp; slot < TB; slot += n_warps) {
            const long long t = batch * TB + slot;
            mask_t* M = sM + slot * A;
            if (lane < A) M[lane] = PM::zero();
            long long lo = 0, hi = 0;
            if (t < P.n_traces && lane == 0) { const long long tr = row_trace<WL>(P, t); lo = P.trace_off[tr]; hi = P.trace_off[tr + 1]; }
            lo = shfl64(lo, 0);
            hi = shfl64(hi, 0);
            const int len = (int)(hi - lo);
            __syncwarp();
            uint32_t* Mw = reinterpret_cast<uint32_t*>(M);  // word w of activity x at [x * STORE + w]
            int px = -1;  // activity of the event before this chunk
            for (int base = 0; base < len; base += 32) {
                const int x = base + lane < len ? __ldg(P.act + lo + base + lane) : -1;
                const bool valid = x >= 0 && x < A;
                const unsigned grp = __match_any_sync(0xffffffffu, x);
                if (valid && lane == __ffs(grp) - 1) Mw[x * PM::STORE + (base >> 5)] = grp;
                // chain pairs (countResponseChain :83-89 = countPrecedenceChain :96-102): adjacent events a b, a != b
                int prev = __shfl_up_sync(0xffffffffu, x, 1);
                if (lane == 0) prev = px;
                const bool pvalid = prev >= 0 && prev < A;
                if (valid && pvalid && prev != x) atomicAdd(&s_chain[prev * A + x], 1u);
                px = __shfl_sync(0xffffffffu, x, 31);
                if (base == 0 && lane == 0 && valid) atomicAdd(&s_first[x], 1u);                 // QueryPlanPositions :51-79
                if (base + 32 >= len && lane == ((len - 1) & 31) && valid) atomicAdd(&s_last[x], 1u);
            }
            __syncwarp();
            if (len > 0) ++w_nonempty;
            if (lane < A) {
                const mask_t m = M[lane];
                const int cnt = PM::popc(m);
                sBL[slot * A + lane] = PM::below_last(m);
                sAF[slot * A + lane] = PM::above_first(m);
                if (cnt) {
                    a_tot += cnt;
                    ++a_uniq;
                    if (cnt >= 2) ++a_diag;
                    if (cnt > P.k_cap) ++w_hist_ovf;
                    else if (cnt < HS) atomicAdd(&s_hist[lane * HS + cnt], 1u);
                    else atomicAdd(o_hist + (long long)lane * (P.k_cap + 1) + cnt, sgn<WL>(P, 1ull));
                }
            }
        }
        __syncthreads();
        // ---------------------------------------------------------------- phase 2: one thread per activity pair
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (pa[j] < 0) continue;
            const int a = pa[j], b = pb[j];
#pragma unroll 2
            for (int slot = 0; slot < TB; ++slot) {
                const mask_t Ma = sM[slot * A + a], Mb = sM[slot * A + b];
                const mask_t BLa = sBL[slot * A + a], BLb = sBL[slot * A + b];
                const mask_t AFa = sAF[slot * A + a], AFb = sAF[slot * A + b];
                const int r_ab = PM::popc_and(Ma, BLb), r_ba = PM::popc_and(Mb, BLa);
                c_r_ab[j] += r_ab;
                c_r_ba[j] += r_ba;
                c_p_ab[j] += PM::popc_and(Mb, AFa);
                c_p_ba[j] += PM::popc_and(Ma, AFb);
                c_ord_ab[j] += r_ab != 0;
                c_ord_ba[j] += r_ba != 0;
                c_co[j] += (r_ab | r_ba) != 0;
                c_alt_ab[j] += PM::alt(Ma, Mb);
                c_alt_ba[j] += PM::alt(Mb, Ma);
            }
        }
        __syncthreads();
        // 32-bit counters: a pair gains at most 32 * NW per trace
        if (++since_flush >= (1 << 24) / (TB * 32 * NW)) { flush_pairs(); since_flush = 0; }
    }
    flush_pairs();
    if (lane < A) {
        if (a_tot) atomicAdd(o_tot + lane, sgn<WL>(P, a_tot));
        if (a_uniq) atomicAdd(o_uniq + lane, sgn<WL>(P, a_uniq));
        if (a_diag) { atomicAdd(o_co + (long long)lane * A + lane, sgn<WL>(P, a_diag)); atomicAdd(o_ord + (long long)lane * A + lane, sgn<WL>(P, a_diag)); }
    }
    if (lane == 0) {
        if (w_nonempty) atomicAdd(&s_misc[1], w_nonempty);
    }
    if (w_hist_ovf) atomicAdd(&s_misc[0], w_hist_ovf);
    __syncthreads();
    for (int i = threadIdx.x; i < A; i += blockDim.x) {
        if (s_first[i]) atomicAdd(o_first + i, sgn<WL>(P, s_first[i]));
        if (s_last[i]) atomicAdd(o_last + i, sgn<WL>(P, s_last[i]));
    }
    for (int i = threadIdx.x; i < A * HS; i += blockDim.x) {
        const int a = i / HS, k = i % HS;
        if (s_hist[i] && k <= P.k_cap) atomicAdd(o_hist + (long long)a * (P.k_cap + 1) + k, sgn<WL>(P, s_hist[i]));
    }
    for (int i = threadIdx.x; i < AA; i += blockDim.x)
        if (s_chain[i]) {
            atomicAdd(o_chain_r + i, sgn<WL>(P, s_chain[i]));
            atomicAdd(o_chain_p + i, sgn<WL>(P, s_chain[i]));
        }
    if (threadIdx.x == 0) {
        if (s_misc[0]) atomicAdd(o_prec + 5ll * AA, sgn<WL>(P, s_misc[0]));
        if (s_misc[1]) atomicAdd(o_prec + 5ll * AA + 1, sgn<WL>(P, s_misc[1]));
    }
}

// ---------------------------------------------------------------------------------- K3 for ANY alphabet and trace length
// More than MAX_A_SMEM activities: the A x A matrices no longer fit in shared memory, and a trace only ever holds a small
// part of the alphabet.  One warp per trace; the warp keeps its per-activity state (count, first, last, slot) and the list
// of the trace's DISTINCT activities (with running count and last position per slot) in a private slice of a global scratch
// (plain loads / stores: the slice is only touched by this warp), and every loop that was "lanes = activities" in the
// kernels above becomes "lanes = distinct activities of this trace".  Counts go to the output with 64-bit atomics.  Same
// definitions, same order of the serial pass: pass 1 counts, pass 2 existence + presence, pass 3 response / precedence at
// the first / last occurrences, alternate at every event, chain on adjacent events.
struct DeclareAnyParams {
    DeclareParams d;
    uint32_t* scratch;   // [warps][7][A]
};

template <bool WL>
__global__ void __launch_bounds__(DT) declare_any_kernel(const __grid_constant__ DeclareAnyParams Q) {
    const DeclareParams& P = Q.d;
    const int A = P.A;
    const long long AA = (long long)A * A;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long gw = (long long)blockIdx.x * (DT / 32) + warp, warps_total = (long long)gridDim.x * (DT / 32);
    uint32_t* w_cnt = Q.scratch + gw * 7 * A;   // zero outside a trace
    uint32_t* w_first = w_cnt + A;
    uint32_t* w_last = w_first + A;
    uint32_t* w_slot = w_last + A;              // activity -> slot in the distinct list
    uint32_t* w_act = w_slot + A;               // slot -> activity
    uint32_t* w_run = w_act + A;                // slot -> occurrences so far (pass 3)
    int* w_lastpos = reinterpret_cast<int*>(w_run + A);   // slot -> last position so far (pass 3)

    unsigned long long* o_tot = P.out;
    unsigned long long* o_uniq = o_tot + A;
    unsigned long long* o_first = o_uniq + A;
    unsigned long long* o_last = o_first + A;
    unsigned long long* o_hist = o_last + A;
    unsigned long long* o_co = o_hist + (long long)A * (P.k_cap + 1);
    unsigned long long* o_ord = o_co + AA;
    unsigned long long* o_resp = o_ord + AA;
    unsigned long long* o_prec = o_resp + AA;
    unsigned long long* o_alt = o_prec + AA;          // alternate response; the precedence copy is made by the host call
    unsigned long long* o_chain = o_alt + 2 * AA;     // chain response; likewise

    unsigned long long n_nonempty = 0, n_hist_ovf = 0;
    for (long long t = gw; t < P.n_traces; t += warps_total) {
        long long lo = 0, hi = 0;
        if (lane == 0) { const long long tr = row_trace<WL>(P, t); lo = P.trace_off[tr]; hi = P.trace_off[tr + 1]; }
        lo = shfl64(lo, 0);
        hi = shfl64(hi, 0);
        if (hi <= lo) continue;
        const long long len = hi - lo;
        ++n_nonempty;
        // pass 1: count / first / last per activity, list of distinct activities (in order of first occurrence)
        int d = 0;
        for (long long base = 0; base < len; base += 32) {
            const int x = base + lane < len ? __ldg(P.act + lo + base + lane) : -1;
            const bool valid = x >= 0 && x < A;
            const unsigned grp = __match_any_sync(0xffffffffu, valid ? x : A + lane);
            const bool leader = valid && lane == __ffs(grp) - 1;
            uint32_t c = 0;
            if (leader) c = w_cnt[x];
            const bool is_new = leader && c == 0;
            const unsigned nb = __ballot_sync(0xffffffffu, is_new);
            if (leader) {
                if (is_new) {
                    const int sl = d + __popc(nb & ((1u << lane) - 1u));
                    w_first[x] = (uint32_t)(base + lane);
                    w_slot[x] = (uint32_t)sl;
                    w_act[sl] = (uint32_t)x;
                    w_run[sl] = 0;
                    w_lastpos[sl] = -1;
                }
                w_cnt[x] = c + (uint32_t)__popc(grp);
                w_last[x] = (uint32_t)(base + 31 - __clz(grp));
            }
            d += __popc(nb);
            __syncwarp();
        }
        if (lane == 0) {
            const int xf = __ldg(P.act + lo), xl = __ldg(P.act + hi - 1);
            if (xf >= 0 && xf < A) atomicAdd(o_first + xf, sgn<WL>(P, 1ull));
            if (xl >= 0 && xl < A) atomicAdd(o_last + xl, sgn<WL>(P, 1ull));
        }
        // pass 2: existence counts and the presence matrices
        for (int j = lane; j < d; j += 32) {
            const int b = (int)w_act[j];
            const uint32_t c = w_cnt[b];
            atomicAdd(o_tot + b, sgn<WL>(P, c));
            atomicAdd(o_uniq + b, sgn<WL>(P, 1ull));
            if (c > (uint32_t)P.k_cap) ++n_hist_ovf;
            else atomicAdd(o_hist + (long long)b * (P.k_cap + 1) + c, sgn<WL>(P, 1ull));
            if (c >= 2) { atomicAdd(o_ord + (long long)b * A + b, sgn<WL>(P, 1ull)); atomicAdd(o_co + (long long)b * A + b, sgn<WL>(P, 1ull)); }
        }
        for (int ai = 0; ai < d; ++ai) {
            const int a = (int)w_act[ai];
            const uint32_t fa = w_first[a];
            for (int j = lane; j < d; j += 32) {
                if (j == ai) continue;
                const int b = (int)w_act[j];
                atomicAdd(o_co + (long long)a * A + b, sgn<WL>(P, 1ull));
                if (fa < w_last[b]) atomicAdd(o_ord + (long long)a * A + b, sgn<WL>(P, 1ull));
            }
        }
        // pass 3: serial over the events
        int px = -1;
        for (long long base = 0; base < len; base += 32) {
            const int mine = base + lane < len ? __ldg(P.act + lo + base + lane) : -1;
            const int n_here = len - base < 32 ? (int)(len - base) : 32;
            for (int k = 0; k < n_here; ++k) {
                const int x = __shfl_sync(0xffffffffu, mine, k);
                const long long i = base + k;
                if (x < 0 || x >= A) { px = -1; continue; }
                const int sx = (int)w_slot[x];
                const bool is_last = w_last[x] == (uint32_t)i, is_first = w_first[x] == (uint32_t)i;
                const int prev = w_lastpos[sx];
                for (int j = lane; j < d; j += 32) {
                    if (j == sx) continue;
                    const int o = (int)w_act[j];
                    const uint32_t r = w_run[j];
                    if (is_last && r) atomicAdd(o_resp + (long long)o * A + x, sgn<WL>(P, r));                       // response[o][x]
                    if (is_first) {
                        const uint32_t co = w_cnt[o];
                        if (co > r) atomicAdd(o_prec + (long long)x * A + o, sgn<WL>(P, (co - r)));                  // precedence[x][o]
                    }
                    if (w_lastpos[j] > prev) atomicAdd(o_alt + (long long)o * A + x, sgn<WL>(P, 1ull));                                  // alternate[o][x]
                }
                __syncwarp();
                if (lane == 0) {
                    w_run[sx] += 1;
                    w_lastpos[sx] = (int)i;
                    if (px >= 0 && px != x) atomicAdd(o_chain + (long long)px * A + x, sgn<WL>(P, 1ull));
                }
                px = x;
                __syncwarp();
            }
        }
        for (int j = lane; j < d; j += 32) w_cnt[w_act[j]] = 0;
        __syncwarp();
    }
    if (lane == 0 && n_nonempty) atomicAdd(o_prec + 5 * AA + 1, sgn<WL>(P, n_nonempty));
    if (n_hist_ovf) atomicAdd(o_prec + 5 * AA, sgn<WL>(P, n_hist_ovf));
}

// longest trace of the log, or (WL) of the traces work[0 .. n_traces)
template <bool WL>
__global__ void max_trace_len_kernel(const int64_t* trace_off, const int64_t* work, int64_t n_traces, unsigned long long* out) {
    unsigned long long m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_traces; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = WL ? work[i] : i;
        const long long d = trace_off[t + 1] - trace_off[t];
        if (d > 0 && (unsigned long long)d > m) m = (unsigned long long)d;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        const unsigned long long y = __shfl_xor_sync(0xffffffffu, m, d);
        m = y > m ? y : m;
    }
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

template <int NW, int PPT, bool WL>
static int launch_pairs(const Ctx* ctx, cudaStream_t stream, const DeclareParams& P, int threads) {
    const int A = P.A;
    const size_t smem = (size_t)3 * TB * A * sizeof(typename PosMask<NW>::T) + sizeof(uint32_t) * ((size_t)A * A + 2 * A + (size_t)A * HS);
    auto kern = declare_pairs_kernel<NW, PPT, WL>;
    SIESTA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    SIESTA_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) per_sm = 1;
    const int64_t n_batches = (P.n_traces + TB - 1) / TB;
    int grid = (int)std::min<int64_t>(std::max<int64_t>(n_batches, 1), (int64_t)ctx->sm_count * per_sm);
    kern<<<grid, threads, smem, stream>>>(P);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

// CTA size of a serial kernel: the one that keeps the most warps resident.  The count matrices live in shared memory per
// CTA, so a large alphabet fits one CTA per SM, and that CTA has to bring all of the SM's warps (256 threads left 8 warps on
// an SM at 100 activities).
template <class K, class SmemOf>
static int pick_cta(K kern, SmemOf smem_of, int* threads, size_t* smem, int* per_sm) {
    int best_warps = 0;
    for (int dt : {256, 512, DTS_MAX}) {
        const size_t sm = smem_of(dt);
        if (sm > (size_t)227 * 1024) continue;
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, dt, sm) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        if (n * (dt / 32) > best_warps) {
            best_warps = n * (dt / 32);
            *threads = dt;
            *smem = sm;
            *per_sm = n;
        }
    }
    if (!best_warps) {
        set_error("declare counting: no CTA size fits the shared memory of this alphabet");
        return SIESTA_E_UNSUPPORTED;
    }
    SIESTA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    return SIESTA_OK;
}

template <int NB, bool WL>
static int launch_alt_chain(const Ctx* ctx, cudaStream_t stream, const DeclareParams& P) {
    auto kern = declare_alt_chain_kernel<NB, WL>;
    int dt = 0, per_sm = 0;
    size_t smem = 0;
    const int A = P.A;
    int rc = pick_cta(kern, [A](int) { return sizeof(uint32_t) * (size_t)2 * A * A; }, &dt, &smem, &per_sm);
    if (rc) return rc;
    const int64_t ctas_needed = (P.n_traces + dt / 32 - 1) / (dt / 32);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(ctas_needed, 1), (int64_t)ctx->sm_count * per_sm);
    kern<<<grid, dt, smem, stream>>>(P);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

static size_t declare_smem(int A, int dt) { return sizeof(uint32_t) * ((size_t)4 * A * A + 4 * A + (size_t)A * HS + (size_t)(dt / 32) * 3 * A); }

template <int NB, bool WL>
static int launch_declare(const Ctx* ctx, cudaStream_t stream, const DeclareParams& P) {
    auto kern = declare_kernel<NB, WL>;
    int dt = 0, per_sm = 0;
    size_t smem = 0;
    const int A = P.A;
    int rc = pick_cta(kern, [A](int t) { return declare_smem(A, t); }, &dt, &smem, &per_sm);
    if (rc) return rc;
    const int64_t ctas_needed = (P.n_traces + dt / 32 - 1) / (dt / 32);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(ctas_needed, 1), (int64_t)ctx->sm_count * per_sm);
    kern<<<grid, dt, smem, stream>>>(P);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

// declare_any_kernel runs for alphabets above MAX_A_SMEM, or for any alphabet under SIESTA_K3_ANY
static bool k3_any(int A) { return A > MAX_A_SMEM || std::getenv("SIESTA_K3_ANY") != nullptr; }

// The kernels that keep the count matrices in shared memory (at most MAX_A_SMEM activities): the pair kernel when the
// alphabet has at most 32 activities and the longest trace of the launch at most 128 events (its mask width follows that
// length), the serial kernels otherwise.  Counts are added to P.out.
template <bool WL>
static int launch_smem_family(const Ctx* ctx, cudaStream_t stream, const DeclareParams& P, int64_t max_len) {
    const int A = P.A;
    int rc = SIESTA_OK;
    if (A <= 32 && max_len <= 128 && std::getenv("SIESTA_K3_SERIAL") == nullptr) {
        // one kernel: position masks + pair-owned counters
        const int n_pairs = A * (A - 1) / 2;
        const int ppt = n_pairs > 256 ? 2 : 1;
        const int threads = std::max(32, std::min(256, ((ppt == 1 ? n_pairs : (n_pairs + 1) / 2) + 31) / 32 * 32));
        if (max_len <= 64) rc = ppt == 1 ? launch_pairs<2, 1, WL>(ctx, stream, P, threads) : launch_pairs<2, 2, WL>(ctx, stream, P, threads);
        else if (max_len <= 96) rc = ppt == 1 ? launch_pairs<3, 1, WL>(ctx, stream, P, threads) : launch_pairs<3, 2, WL>(ctx, stream, P, threads);
        else rc = ppt == 1 ? launch_pairs<4, 1, WL>(ctx, stream, P, threads) : launch_pairs<4, 2, WL>(ctx, stream, P, threads);
        return rc;
    }
    const int nb = (A + 31) / 32;
    if (nb == 1) rc = launch_declare<1, WL>(ctx, stream, P);
    else if (nb == 2) rc = launch_declare<2, WL>(ctx, stream, P);
    else if (nb == 3) rc = launch_declare<3, WL>(ctx, stream, P);
    else rc = launch_declare<4, WL>(ctx, stream, P);
    if (rc) return rc;
    if (nb == 1) rc = launch_alt_chain<1, WL>(ctx, stream, P);
    else if (nb == 2) rc = launch_alt_chain<2, WL>(ctx, stream, P);
    else if (nb == 3) rc = launch_alt_chain<3, WL>(ctx, stream, P);
    else rc = launch_alt_chain<4, WL>(ctx, stream, P);
    return rc;
}

// Grid of declare_any_kernel for `rows` rows: two CTAs per SM (the kernel is bound by the 64-bit atomics on the result;
// more resident warps were measured slower, 86.7 against 82.7 ms per 1e8 events at 400 activities)
static int any_grid(const Ctx* ctx, int64_t rows) {
    const int64_t ctas_needed = (rows + DT / 32 - 1) / (DT / 32);
    return (int)std::min<int64_t>(std::max<int64_t>(ctas_needed, 1), (int64_t)ctx->sm_count * 2);
}
static size_t any_scratch_bytes(int grid, int A) { return sizeof(uint32_t) * (size_t)grid * (DT / 32) * 7 * A; }

// the scratch must be zero at the launch; the kernel leaves it zero
template <bool WL>
static cudaError_t launch_any(cudaStream_t stream, const DeclareParams& P, int grid, void* scratch) {
    DeclareAnyParams Q;
    Q.d = P;
    Q.scratch = reinterpret_cast<uint32_t*>(scratch);
    declare_any_kernel<WL><<<grid, DT, 0, stream>>>(Q);
    SIESTA_LAUNCHED();
    return cudaGetLastError();
}

// declare_any_kernel writes the response copies of the alternate and chain matrices; the precedence copies are equal
static cudaError_t any_twin_copies(int64_t* d_out, int A, int k_cap, cudaStream_t stream) {
    const size_t aa = sizeof(int64_t) * (size_t)A * A;
    int64_t* o_alt = d_out + 4ll * A + (int64_t)A * (k_cap + 1) + 4ll * A * A;
    cudaError_t e = cudaMemcpyAsync(o_alt + (size_t)A * A, o_alt, aa, cudaMemcpyDeviceToDevice, stream);                      // alternate precedence = response
    if (e == cudaSuccess) e = cudaMemcpyAsync(o_alt + 3 * (size_t)A * A, o_alt + 2 * (size_t)A * A, aa, cudaMemcpyDeviceToDevice, stream);  // chain likewise
    return e;
}

// ------------------------------------------------------------------------------------------ refresh after a log append
// Every block of the packed result is a sum of per-trace contributions, and an append changes only the traces it lists:
//     counts(new log) = remap(counts(old log)) - K3(old log, listed old traces) + K3(new log, listed traces)
// in wrapping 64-bit arithmetic (remap moves the blocks from the old alphabet to the new one, new rows and columns zero).
// Both work-list launches use the new alphabet and accumulate into one delta in the new layout; declare_merge_kernel adds
// it to the remapped old counts.

// Unlisted traces must keep their length (the cheap guard against a wrong trace_idx):
//     bad = #{t < T : length differs} - #{listed t < T : length differs}
__global__ void refresh_check_kernel(const int64_t* __restrict__ old_off, const int64_t* __restrict__ new_off, int64_t T,
                                     const int64_t* __restrict__ work, int64_t n_old, unsigned long long* bad) {
    long long c = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t t = i0; t < T; t += stride) c += (old_off[t + 1] - old_off[t]) != (new_off[t + 1] - new_off[t]);
    for (int64_t i = i0; i < n_old; i += stride) {
        const int64_t t = work[i];
        c -= (old_off[t + 1] - old_off[t]) != (new_off[t + 1] - new_off[t]);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(bad, (unsigned long long)c);
}

// out = old moved from alphabet A0 to A1 (zero in the new rows and columns) + delta: one coalesced pass over the new layout.
// out may be old (A0 == A1) or delta: every element is read and written by the same thread.
__global__ void declare_merge_kernel(const unsigned long long* old, int A0, int A1, int64_t K, int64_t n, const unsigned long long* delta,
                                     unsigned long long* out) {
    const int64_t h0 = 4ll * A1, m0 = h0 + (int64_t)A1 * K, s0 = m0 + 8ll * A1 * A1;   // hist, matrices, scalars (new layout)
    const int64_t oh0 = 4ll * A0, om0 = oh0 + (int64_t)A0 * K;                          // same, old layout
    const int64_t AA1 = (int64_t)A1 * A1, AA0 = (int64_t)A0 * A0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t src = i;
        if (A0 != A1) {
            if (i < h0) {   // tot uniq first last
                const int64_t blk = i / A1, a = i - blk * A1;
                src = a < A0 ? blk * A0 + a : -1;
            } else if (i < m0) {   // hist[a][k]
                const int64_t a = (i - h0) / K, k = (i - h0) - a * K;
                src = a < A0 ? oh0 + a * K + k : -1;
            } else if (i < s0) {   // eight [a][b] matrices
                const int64_t j = i - m0, m = j / AA1, r = j - m * AA1, a = r / A1, b = r - a * A1;
                src = a < A0 && b < A0 ? om0 + m * AA0 + a * A0 + b : -1;
            } else {   // hist_overflow, n_nonempty
                src = om0 + 8 * AA0 + (i - s0);
            }
        }
        out[i] = (src >= 0 ? old[src] : 0ull) + delta[i];
    }
}

bool declare_refresh_check_host(const char* fn, const Log* O, const Log* N, const int64_t* trace_idx, int64_t n_listed, int32_t k_cap) {
    if (n_listed < 0 || (n_listed > 0 && !trace_idx)) {
        set_error(std::string(fn) + ": null argument");
        return false;
    }
    if (k_cap < 1) {
        set_error(std::string(fn) + ": k_cap must be >= 1");
        return false;
    }
    if (O->ctx != N->ctx) {
        set_error(std::string(fn) + ": the two logs are on different contexts");
        return false;
    }
    if (O->d_src_event || N->d_src_event || O->n_blocks > 0 || N->n_blocks > 0) {
        set_error(std::string(fn) + ": derived (filter / group) and block-cyclic logs are not refreshed");
        return false;
    }
    if (N->n_traces < O->n_traces || N->n_activities < O->n_activities) {
        set_error(std::string(fn) + ": new_log has fewer traces or a smaller alphabet than old_log");
        return false;
    }
    const int64_t T = O->n_traces, T2 = N->n_traces;
    int64_t n_new = 0;
    for (int64_t i = 0; i < n_listed; ++i) {
        if (trace_idx[i] < 0 || trace_idx[i] >= T2 || (i > 0 && trace_idx[i] <= trace_idx[i - 1])) {
            set_error(std::string(fn) + ": trace_idx must ascend strictly inside [0, new_log's n_traces)");
            return false;
        }
        n_new += trace_idx[i] >= T;
    }
    if (n_new != T2 - T) {
        set_error(std::string(fn) + ": trace_idx must list every trace new_log adds (as passed to siesta_log_append)");
        return false;
    }
    return true;
}

// Old ids outside the old alphabet that the new one covers: unlisted traces may gain counted events
bool declare_refresh_needs_full(const Log* O, const Log* N) { return !O->act_valid && N->n_activities > O->n_activities; }

// After declare_refresh_check_host: the listed traces go to the device, one pass over both offset arrays checks the
// unlisted traces' lengths, and (pair-kernel alphabets) the longest listed trace of each log is measured; one 24-byte read.
int declare_refresh_stage(const char* fn, DeclareRefresh* r, const int64_t* trace_idx, cudaStream_t stream, cudaEvent_t copied) {
    Log* O = r->O;
    Log* N = r->N;
    Ctx* c = N->ctx;
    r->n_old = (int64_t)(std::lower_bound(trace_idx, trace_idx + r->n_listed, O->n_traces) - trace_idx);
    const size_t wbytes = ((size_t)std::max<int64_t>(r->n_listed, 1) * 8 + 255) & ~(size_t)255;
    r->block = dev_arena_alloc(c, wbytes + 256);
    if (!r->block) return SIESTA_E_NOMEM;
    r->d_work = reinterpret_cast<int64_t*>(r->block);
    unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(static_cast<char*>(r->block) + wbytes);   // bad, max old, max new
    SIESTA_CUDA_OK(cudaMemsetAsync(d_cnt, 0, 24, stream));
    if (r->n_listed) SIESTA_CUDA_OK(cudaMemcpyAsync(r->d_work, trace_idx, (size_t)r->n_listed * 8, cudaMemcpyHostToDevice, stream));
    if (copied) SIESTA_CUDA_OK(cudaEventRecord(copied, stream));
    const int64_t T = O->n_traces;
    if (T > 0) {
        refresh_check_kernel<<<(unsigned)std::min<int64_t>((T + 255) / 256, 4 * c->sm_count), 256, 0, stream>>>(O->d_trace_off, N->d_trace_off, T,
                                                                                                           r->d_work, r->n_old, d_cnt);
        SIESTA_LAUNCHED();
    }
    if (N->n_activities <= 32 && !k3_any(N->n_activities)) {
        if (r->n_old > 0) {
            max_trace_len_kernel<true><<<(unsigned)std::min<int64_t>((r->n_old + 255) / 256, 4 * c->sm_count), 256, 0, stream>>>(O->d_trace_off, r->d_work,
                                                                                                                           r->n_old, d_cnt + 1);
            SIESTA_LAUNCHED();
        }
        if (r->n_listed > 0) {
            max_trace_len_kernel<true><<<(unsigned)std::min<int64_t>((r->n_listed + 255) / 256, 4 * c->sm_count), 256, 0, stream>>>(N->d_trace_off, r->d_work,
                                                                                                                              r->n_listed, d_cnt + 2);
            SIESTA_LAUNCHED();
        }
    }
    SIESTA_CUDA_OK(cudaGetLastError());
    unsigned long long h[3] = {0, 0, 0};
    SIESTA_CUDA_OK(cudaMemcpyAsync(h, d_cnt, 24, cudaMemcpyDeviceToHost, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    r->max_old = (int64_t)h[1];
    r->max_new = (int64_t)h[2];
    if (h[0]) {
        set_error(std::string(fn) + ": " + std::to_string(h[0]) +
                  " unlisted trace(s) differ in length between the two logs (trace_idx must be what siesta_log_append was given)");
        return SIESTA_E_INVALID;
    }
    return SIESTA_OK;
}

// d_delta (new layout) = K3(new log, listed) - K3(old log, listed old traces); enqueued on `stream`
int declare_refresh_delta(DeclareRefresh* r, int32_t k_cap, int64_t* d_delta, cudaStream_t stream) {
    Log* O = r->O;
    Log* N = r->N;
    const int A = N->n_activities;
    SIESTA_CUDA_OK(cudaMemsetAsync(d_delta, 0, sizeof(int64_t) * (size_t)siesta_declare_counts_size(A, k_cap), stream));
    DeclareParams P;
    P.act = nullptr;
    P.A = A;
    P.k_cap = k_cap;
    P.out = reinterpret_cast<unsigned long long*>(d_delta);
    P.work = r->d_work;
    DeclareParams Pold = P, Pnew = P;
    Pold.trace_off = O->d_trace_off;
    Pold.act = O->d_act;
    Pold.n_traces = r->n_old;
    Pold.neg = 1;
    Pnew.trace_off = N->d_trace_off;
    Pnew.act = N->d_act;
    Pnew.n_traces = r->n_listed;
    Pnew.neg = 0;
    if (k3_any(A)) {
        const int grid = std::max(any_grid(N->ctx, r->n_old), any_grid(N->ctx, r->n_listed));
        const size_t sbytes = any_scratch_bytes(grid, A);
        r->scratch = dev_arena_alloc(N->ctx, sbytes);
        if (!r->scratch) return SIESTA_E_NOMEM;
        SIESTA_CUDA_OK(cudaMemsetAsync(r->scratch, 0, sbytes, stream));
        cudaError_t e = cudaSuccess;
        if (r->n_old > 0) e = launch_any<true>(stream, Pold, any_grid(N->ctx, r->n_old), r->scratch);
        if (e == cudaSuccess && r->n_listed > 0) e = launch_any<true>(stream, Pnew, any_grid(N->ctx, r->n_listed), r->scratch);
        if (e == cudaSuccess) e = any_twin_copies(d_delta, A, k_cap, stream);
        if (e != cudaSuccess) {
            set_error(std::string("declare_any_kernel: ") + cudaGetErrorString(e));
            return SIESTA_E_CUDA;
        }
        return SIESTA_OK;
    }
    int rc = SIESTA_OK;
    if (r->n_old > 0) rc = launch_smem_family<true>(N->ctx, stream, Pold, r->max_old);
    if (rc == SIESTA_OK && r->n_listed > 0) rc = launch_smem_family<true>(N->ctx, stream, Pnew, r->max_new);
    return rc;
}

int declare_merge(const int64_t* d_old, int32_t A0, int32_t A1, int32_t k_cap, const int64_t* d_delta, int64_t* d_out, const Ctx* c,
                  cudaStream_t stream) {
    const int64_t n = siesta_declare_counts_size(A1, k_cap);
    declare_merge_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 8 * c->sm_count), 256, 0, stream>>>(
        reinterpret_cast<const unsigned long long*>(d_old), A0, A1, (int64_t)k_cap + 1, n, reinterpret_cast<const unsigned long long*>(d_delta),
        reinterpret_cast<unsigned long long*>(d_out));
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

// returns the arena blocks once nothing on `stream` uses them
void declare_refresh_release(DeclareRefresh* r, cudaStream_t stream) {
    if (!r->block && !r->scratch) return;
    cudaStreamSynchronize(stream);
    if (r->block) dev_arena_free(r->N->ctx, r->block);
    if (r->scratch) dev_arena_free(r->N->ctx, r->scratch);
    r->block = r->scratch = nullptr;
}

}  // namespace siesta

using namespace siesta;

extern "C" int64_t siesta_declare_counts_size(int32_t A, int32_t k_cap) {
    return 4ll * A + (int64_t)A * (k_cap + 1) + 8ll * A * A + 2;
}

extern "C" int siesta_declare_counts_device(siesta_log* log, int32_t k_cap, int64_t* d_out, void* stream_, double* kernel_ms) {
    if (!log || !d_out || k_cap < 1) {
        set_error("siesta_declare_counts_device: bad argument");
        return SIESTA_E_INVALID;
    }
    Log* L = reinterpret_cast<Log*>(log);
    const int A = L->n_activities;
    if (A < 1 || A > MAX_A_ANY) {
        set_error("declare counting: 1 <= n_activities <= " + std::to_string(MAX_A_ANY) + " (the eight A x A count matrices of the result)");
        return SIESTA_E_UNSUPPORTED;
    }
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    cudaStream_t stream = stream_ ? reinterpret_cast<cudaStream_t>(stream_) : L->ctx->stream;
    DeclareParams P;
    P.trace_off = L->d_trace_off;
    P.act = L->d_act;
    P.n_traces = L->n_traces;
    P.A = A;
    P.k_cap = k_cap;
    P.out = reinterpret_cast<unsigned long long*>(d_out);
    P.work = nullptr;
    P.neg = 0;
    cudaEvent_t e0, e1;
    SIESTA_CUDA_OK(cudaEventCreate(&e0));
    SIESTA_CUDA_OK(cudaEventCreate(&e1));
    SIESTA_CUDA_OK(cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)siesta_declare_counts_size(A, k_cap), stream));
    int rc = SIESTA_OK;
    // exact length of the longest trace (the caller's hint is not trusted); cached on the log
    if (L->true_max_len < 0) {
        unsigned long long* d_max = nullptr;
        SIESTA_CUDA_OK(cudaMallocAsync((void**)&d_max, 8, stream));
        SIESTA_CUDA_OK(cudaMemsetAsync(d_max, 0, 8, stream));
        if (L->n_traces > 0) {
            max_trace_len_kernel<false><<<(unsigned)std::min<int64_t>((L->n_traces + 255) / 256, 4 * L->ctx->sm_count), 256, 0, stream>>>(
                L->d_trace_off, nullptr, L->n_traces, d_max);
            SIESTA_LAUNCHED();
        }
        unsigned long long h_max = 0;
        SIESTA_CUDA_OK(cudaMemcpyAsync(&h_max, d_max, 8, cudaMemcpyDeviceToHost, stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
        cudaFreeAsync(d_max, stream);
        L->true_max_len = (int64_t)h_max;
    }
    SIESTA_CUDA_OK(cudaEventRecord(e0, stream));
    if (k3_any(A)) {
        // any alphabet, any trace length: lanes = the distinct activities of a trace, counts by 64-bit atomics
        const int grid = any_grid(L->ctx, L->n_traces);
        const size_t sbytes = any_scratch_bytes(grid, A);
        void* scratch = dev_arena_alloc(L->ctx, sbytes);
        if (!scratch) return SIESTA_E_NOMEM;
        SIESTA_CUDA_OK(cudaMemsetAsync(scratch, 0, sbytes, stream));
        cudaError_t e = launch_any<false>(stream, P, grid, scratch);
        if (e == cudaSuccess) e = any_twin_copies(d_out, A, k_cap, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        dev_arena_free(L->ctx, scratch);
        if (e != cudaSuccess) {
            set_error(std::string("declare_any_kernel: ") + cudaGetErrorString(e));
            return SIESTA_E_CUDA;
        }
    } else {
        rc = launch_smem_family<false>(L->ctx, stream, P, L->true_max_len);
        if (rc) return rc;
    }
    SIESTA_CUDA_OK(cudaEventRecord(e1, stream));
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    float ms = 0.f;
    SIESTA_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (kernel_ms) *kernel_ms = ms;
    return SIESTA_OK;
}

extern "C" int siesta_declare_counts(siesta_log* log, int32_t k_cap, int64_t* out, double* kernel_ms) {
    if (!log || !out) {
        set_error("siesta_declare_counts: null argument");
        return SIESTA_E_INVALID;
    }
    Log* L = reinterpret_cast<Log*>(log);
    SIESTA_CUDA_OK(cudaSetDevice(L->ctx->device));
    const size_t bytes = sizeof(int64_t) * (size_t)siesta_declare_counts_size(L->n_activities, k_cap);
    int64_t* d = nullptr;
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d, bytes, L->ctx->stream));
    int rc = siesta_declare_counts_device(log, k_cap, d, L->ctx->stream, kernel_ms);
    if (rc == SIESTA_OK) {
        cudaError_t e = cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, L->ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(L->ctx->stream);
        if (e != cudaSuccess) {
            set_error(std::string("siesta_declare_counts: D2H: ") + cudaGetErrorString(e));
            rc = SIESTA_E_CUDA;
        }
    }
    cudaFreeAsync(d, L->ctx->stream);
    return rc;
}

// ------------------------------------------------------------------------------------------ refresh after a log append
static int refresh_unsupported(const Log* N) {
    if (N->n_activities < 1 || N->n_activities > MAX_A_ANY) {
        set_error("declare counting: 1 <= n_activities <= " + std::to_string(MAX_A_ANY) + " (the eight A x A count matrices of the result)");
        return SIESTA_E_UNSUPPORTED;
    }
    return SIESTA_OK;
}

extern "C" int siesta_declare_counts_refresh_device(siesta_log* old_log, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed,
                                                    int32_t k_cap, const int64_t* d_old, int64_t* d_out, void* stream_, double* kernel_ms) {
    static const char* fn = "siesta_declare_counts_refresh_device";
    Log* O = reinterpret_cast<Log*>(old_log);
    Log* N = reinterpret_cast<Log*>(new_log);
    if (!O || !N || !d_old || !d_out) {
        set_error(std::string(fn) + ": null argument");
        return SIESTA_E_INVALID;
    }
    if (!declare_refresh_check_host(fn, O, N, trace_idx, n_listed, k_cap)) return SIESTA_E_INVALID;
    if (d_out == d_old && N->n_activities != O->n_activities) {
        set_error(std::string(fn) + ": d_out may be d_old only when the alphabet did not grow");
        return SIESTA_E_INVALID;
    }
    if (int rc = refresh_unsupported(N)) return rc;
    SIESTA_CUDA_OK(cudaSetDevice(N->ctx->device));
    cudaStream_t stream = stream_ ? reinterpret_cast<cudaStream_t>(stream_) : N->ctx->stream;
    DeclareRefresh r;
    r.O = O;
    r.N = N;
    r.n_listed = n_listed;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto done = [&](int rc) {
        declare_refresh_release(&r, stream);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        return rc;
    };
    cudaError_t e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    if (e != cudaSuccess) {
        set_error(std::string(fn) + ": " + cudaGetErrorString(e));
        return done(SIESTA_E_CUDA);
    }
    int rc = declare_refresh_stage(fn, &r, trace_idx, stream, e0);   // the time starts after the copy of trace_idx
    if (rc) return done(rc);
    if (declare_refresh_needs_full(O, N)) {   // the header's one fallback: count the new log in full
        done(SIESTA_OK);
        return siesta_declare_counts_device(new_log, k_cap, d_out, stream_, kernel_ms);
    }
    const size_t bytes = sizeof(int64_t) * (size_t)siesta_declare_counts_size(N->n_activities, k_cap);
    void* d_delta = dev_arena_alloc(N->ctx, bytes);
    if (!d_delta) return done(SIESTA_E_NOMEM);
    rc = declare_refresh_delta(&r, k_cap, reinterpret_cast<int64_t*>(d_delta), stream);
    if (rc == SIESTA_OK) rc = declare_merge(d_old, O->n_activities, N->n_activities, k_cap, reinterpret_cast<int64_t*>(d_delta), d_out, N->ctx, stream);
    if (rc == SIESTA_OK) {
        e = cudaEventRecord(e1, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        if (e != cudaSuccess) {
            set_error(std::string(fn) + ": " + cudaGetErrorString(e));
            rc = SIESTA_E_CUDA;
        } else if (kernel_ms) {
            *kernel_ms = ms;
        }
    }
    cudaStreamSynchronize(stream);
    dev_arena_free(N->ctx, d_delta);
    return done(rc);
}

extern "C" int siesta_declare_counts_refresh(siesta_log* old_log, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed, int32_t k_cap,
                                             const int64_t* old_counts, int64_t* out, double* kernel_ms) {
    static const char* fn = "siesta_declare_counts_refresh";
    Log* O = reinterpret_cast<Log*>(old_log);
    Log* N = reinterpret_cast<Log*>(new_log);
    if (!O || !N || !old_counts || !out) {
        set_error(std::string(fn) + ": null argument");
        return SIESTA_E_INVALID;
    }
    // the checks that need no device first: a refused call allocates nothing
    if (!declare_refresh_check_host(fn, O, N, trace_idx, n_listed, k_cap)) return SIESTA_E_INVALID;
    if (int rc = refresh_unsupported(N)) return rc;
    SIESTA_CUDA_OK(cudaSetDevice(N->ctx->device));
    cudaStream_t stream = N->ctx->stream;
    const size_t b_old = sizeof(int64_t) * (size_t)siesta_declare_counts_size(O->n_activities, k_cap);
    const size_t b_new = sizeof(int64_t) * (size_t)siesta_declare_counts_size(N->n_activities, k_cap);
    int64_t* d = nullptr;
    SIESTA_CUDA_OK(cudaMallocAsync((void**)&d, b_old + b_new, stream));
    int64_t* d_old = d;
    int64_t* d_out = d + b_old / sizeof(int64_t);
    cudaError_t e = cudaMemcpyAsync(d_old, old_counts, b_old, cudaMemcpyHostToDevice, stream);
    int rc = e == cudaSuccess ? siesta_declare_counts_refresh_device(old_log, new_log, trace_idx, n_listed, k_cap, d_old, d_out, stream, kernel_ms)
                              : SIESTA_E_CUDA;
    if (e != cudaSuccess) set_error(std::string(fn) + ": H2D: " + cudaGetErrorString(e));
    if (rc == SIESTA_OK) {
        e = cudaMemcpyAsync(out, d_out, b_new, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) {
            set_error(std::string(fn) + ": D2H: " + cudaGetErrorString(e));
            rc = SIESTA_E_CUDA;
        }
    }
    cudaFreeAsync(d, stream);
    return rc;
}
