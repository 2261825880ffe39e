// detect_common.cuh — declarations shared by the translation units of kernel K1 (detect.cu: staged kernel, placement,
// host side; detect_nkp.cu: kernel K1-P).
#pragma once
#include "detect_fast.cuh"

namespace siesta {

constexpr int NT = 128;      // threads per CTA (one warp = one tile of 32 traces)
constexpr int NT_MAX = 128;  // launch bound
// Rows of a trace's shared-memory columns.  The narrow configuration keeps 24 (not 32) so that five CTAs fit beside an
// L1 of ~90 KB (the kernel is sensitive to both, profiles/r01_k1_tuning.md); traces with more relevant events re-run
// on the wide configuration (64 rows, 64-bit masks).
#define ROWS_OF(W) ((W) == 1 ? 24 : 64)

struct DetectParams {
    const int64_t* trace_off;
    const int32_t* act;
    const int64_t* ts_ms;
    const int64_t* cand;      // candidate trace indices or nullptr (= identity)
    const int64_t* work;      // indices into the candidate list to process, or nullptr (= all)
    int64_t n_work;           // number of traces this launch verifies ...
    const unsigned long long* n_work_dev;  // ... or, if set, read from device memory (the narrow launch's overflow count)
    int32_t ovf_slot;         // counter that counts the traces this launch could not hold (4 narrow, 7 wide)
    int32_t tile_slot;        // counter that hands out tiles (16 narrow, 17 wide, 18 K1-P)
    const uint16_t* lut;      // [n_act] smask | fmask << 8
    // alpha_mode 0/1: the pattern's activities are numbered 1..K (K <= 7, "class"); plane p holds, bit-reversed, the
    // activities whose class has bit p set (ids 0..31 in [p][0], 32..63 in [p][1]); cls_word / cls_act give the lut
    // word and the activity id of a class, so the filter needs no table lookup and no re-read of the activity column
    uint32_t relrev[3][2];
    uint16_t cls_word[8];
    int32_t cls_act[8];
    int32_t n_planes;
    int64_t n_events;         // events of the whole log (bound of the vector loads)
    int32_t alpha_mode;       // 0: n_act <= 32, 1: n_act <= 64 (both: ids validated at log load, K <= 7), 2: general (lut in HBM)
    int32_t vec_ok;           // act is 16-byte aligned: 128-bit loads
    int32_t n_act;
    uint32_t flags;
    int32_t needs_ts;
    // dense per-candidate outputs
    uint32_t* d_cnt;          // selected occurrences (0 = no match) | events over the selected occurrences << 16
    int64_t* d_stage;         // staging base (events) of the trace
    int64_t* d_stage_occ;     // staging base (occurrences) of the trace; only with returnAll (else = the candidate's index)
    // staging
    int32_t* s_occ_nev;       // [cap_occ] events per staged occurrence
    int32_t* s_ev_pos;        // [cap_ev]
    int32_t* s_ev_rank;
    int32_t* s_ev_act;
    int64_t* s_ev_ts;
    int64_t cap_occ, cap_ev;
    // K1-P stages at fixed places (no atomic on its critical path): tile i owns the event slots
    // [fix_ev + 32 i fix_np, + 32 fix_np) of a second staging region behind the first one
    int64_t fix_ev;
    int32_t fix_np;
    int64_t fix_occ;          // returnAll: candidate i stages its occurrence's event count at s_occ_nev[fix_occ + i] (-1: not asked for)
    // K1-P, uniform result (one occurrence of fix_np events per matching trace): per tile the lanes that matched
    // (tile_words[tile]) and the lanes sent to the overflow list (tile_words[n_tiles + tile]); each event is staged as
    // one word pos | rank << 8 | act << 16 in s_ev_pos plus its timestamp, and no d_cnt / d_stage is written for the
    // traces K1-P answers.  nullptr: the per-candidate outputs and the four staged columns
    uint32_t* tile_words;
    // K1-P: a state that owns exactly ONE class is the minterm of the class planes with these polarities
    // (st_inv[k][p] = 0 or ~0: plane p enters state k's mask as it is / complemented); st_single[k] = 0: OR of several classes
    uint32_t st_inv[SIESTA_MAX_STATES][3];
    uint8_t st_single[SIESTA_MAX_STATES];
    const uint4* nkp_lut;     // K1-P: [n_act + 1] {m, b0, b1, b2} per activity (detect_nkp.cu), entry n_act = no event
    int32_t tile_batch;       // K1-P: consecutive tiles a warp takes per atomic (one atomic per tile would bound a 10^8-trace scan)
    // counters: 0 occ reserved, 1 ev reserved, 2 emitted, 3 errors, 4 overflow, 5 staging overflow, 6 matched traces,
    // 7 wide overflow, 8-10 phase timing, 13 K1-P overflow; second 128-byte line: 16 / 17 / 18 next tile of the narrow /
    // wide / K1-P launch
    unsigned long long* counters;
    // [3][n_blk] matching traces / occurrences / events per block of 256 candidates, accumulated by the verification
    // kernels themselves (one reduction per tile), so the placement needs no counting pass over the candidates
    unsigned long long* blk_sums;
    int64_t n_blk;
    int64_t* err_list;
    int64_t* ovf_list;
    int64_t ovf_cap;          // entries ovf_list holds (0 = one per candidate); the counter keeps counting past it
};

__device__ __forceinline__ long long shfl_i64(long long v, int src) {
    int lo = __shfl_sync(0xffffffffu, (int)(v & 0xffffffffll), src);
    int hi = __shfl_sync(0xffffffffu, (int)(v >> 32), src);
    return ((long long)hi << 32) | (unsigned int)lo;
}

// status codes of a trace inside the kernel
enum { ST_NONE = 0, ST_MATCH = 1, ST_ERR = 2, ST_OVF = 3 };

// 32 activity ids (four 32-byte sectors, two 128-bit loads each) starting at element e of this lane's trace [o0, o1).
// Sectors past the trace are not touched; the scalar path serves unaligned logs and the last sector of the log.
__device__ __forceinline__ void load_sectors(const DetectParams& P, long long e, long long o0, long long o1, int4 (&v)[8]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const long long c = e + 8 * q;
        if (c >= o1) {
            v[2 * q] = v[2 * q + 1] = make_int4(-1, -1, -1, -1);
        } else if (P.vec_ok && c + 8 <= P.n_events) {
            v[2 * q] = __ldg(reinterpret_cast<const int4*>(P.act + c));
            v[2 * q + 1] = __ldg(reinterpret_cast<const int4*>(P.act + c + 4));
        } else {
            int a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = (c + i < o1 && c + i >= o0) ? __ldg(P.act + c + i) : -1;
            v[2 * q] = make_int4(a[0], a[1], a[2], a[3]);
            v[2 * q + 1] = make_int4(a[4], a[5], a[6], a[7]);
        }
    }
}
// The same for kernel K1-P, which only runs on 32-byte aligned logs with validated activity ids and sends a trace whose
// last sector crosses the end of the log to the staged kernel: no scalar path, a sixth of the code.  Slots outside the
// trace read as activity n_act, the "no event" entry of K1-P's table.
__device__ __forceinline__ void load_sectors_vec(const DetectParams& P, long long e, long long o1, int4 (&v)[8]) {
    const int none = P.n_act;   // the table entry of "no event"
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const long long c = e + 8 * q;
        if (c >= o1) {
            v[2 * q] = v[2 * q + 1] = make_int4(none, none, none, none);
        } else {
            // one 256-bit load = the lane's whole 32-byte sector (sm_100: LDG.E.256); two 128-bit loads would present
            // every sector to the L1 twice
            asm volatile("ld.global.nc.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(v[2 * q].x), "=r"(v[2 * q].y), "=r"(v[2 * q].z), "=r"(v[2 * q].w), "=r"(v[2 * q + 1].x),
                           "=r"(v[2 * q + 1].y), "=r"(v[2 * q + 1].z), "=r"(v[2 * q + 1].w)
                         : "l"(P.act + c));
        }
    }
}

// 16 slots (two sectors) of this lane's trace starting at element e: two 256-bit loads, or "no event" past the trace
__device__ __forceinline__ void load_quarter(const DetectParams& P, long long e, long long o1, int4 (&v)[4]) {
    const int none = P.n_act;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const long long c = e + 8 * q;
        if (c >= o1) {
            v[2 * q] = v[2 * q + 1] = make_int4(none, none, none, none);
        } else {
            asm volatile("ld.global.nc.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(v[2 * q].x), "=r"(v[2 * q].y), "=r"(v[2 * q].z), "=r"(v[2 * q].w), "=r"(v[2 * q + 1].x),
                           "=r"(v[2 * q + 1].y), "=r"(v[2 * q + 1].z), "=r"(v[2 * q + 1].w)
                         : "l"(P.act + c));
        }
    }
}

// Relevance test of the filter: relrev holds the pattern's activity set bit-reversed (bit 31 - a <=> activity a), so
// `relrev << a` moves activity a's bit to the top and one funnel shift pushes it into the survivor mask: two
// instructions per event.  shl.b32 clamps shift amounts above 31, so a masked-out slot (a = -1) pushes 0.
__device__ __forceinline__ uint32_t rel_push32(uint32_t pend, uint32_t relrev, int a) {
    uint32_t t;
    asm("shl.b32 %0, %1, %2;" : "=r"(t) : "r"(relrev), "r"(a));
    return __funnelshift_r(t, pend, 31);
}
// activities 0..31 in relrev_a, 32..63 in relrev_b
__device__ __forceinline__ uint32_t rel_push64(uint32_t pend, uint32_t relrev_a, uint32_t relrev_b, int a) {
    uint32_t t;
    const uint32_t w = ((unsigned)a < 32u) ? relrev_a : (((unsigned)a < 64u) ? relrev_b : 0u);
    asm("shl.b32 %0, %1, %2;" : "=r"(t) : "r"(w), "r"(a & 31));
    return __funnelshift_r(t, pend, 31);
}

// Class bit-planes of 32 consecutive events (bit i = event i), last event first.
template <int NPL, bool WIDE>
__device__ __forceinline__ void scan_block(const DetectParams& P, const int4 (&v)[8], uint32_t (&pl)[3]) {
#pragma unroll
    for (int q = 7; q >= 0; --q) {
        const int a[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
        for (int i = 3; i >= 0; --i) {
#pragma unroll
            for (int p = 0; p < NPL; ++p)
                pl[p] = WIDE ? rel_push64(pl[p], P.relrev[p][0], P.relrev[p][1], a[i]) : rel_push32(pl[p], P.relrev[p][0], a[i]);
        }
    }
}

// EventTs.transformSaseEvent: (int)((t - minTs) / 1000), truncating long division (J/model/Events/EventTs.java:54).
// Differences below 2^32 ms (49 days) take a 32-bit multiply-high instead of the emulated 64-bit division.
__device__ __forceinline__ int rel_seconds(long long diff_ms) {
    if ((unsigned long long)diff_ms < (1ull << 32)) return (int)((uint32_t)diff_ms / 1000u);
    return (int)(diff_ms / 1000);
}

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }


// K1-P launcher (detect_nkp.cu).  space = NKW_RANK / NKW_RAW (nkw_build); tile_batch = tiles a warp takes per atomic.
int launch_nkp(const Ctx* ctx, cudaStream_t stream, const DetectParams& P, const NkwProgram& prog, int space);

}  // namespace siesta
