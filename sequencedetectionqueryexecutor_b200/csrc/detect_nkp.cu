// detect_nkp.cu — kernel K1-P: class NK (no Kleene state) as window walks over one index space (sm_100a).
//
// Replaces, for NFAs of class NK whose first-largest occurrence is asked for and whose predicates read no relative
// seconds, SaseConnector.evaluate + Occurrences.clearOccurrences(false)
// (J/SaseConnection/SaseConnector.java:48-76, J/model/Occurrences.java:58-72); derivation in detect_fast.cuh.
//
// One lane per trace, no per-event loop after the scan:
//   load     the lane streams the trace's 32-byte sectors (<= 64 position slots from the sector of its first event;
//            sixteen 128-bit loads, all issued before the first is used); the offsets of the NEXT tile are requested a
//            tile early, so a tile waits for one memory latency, not two.  (Staging the sectors of tile i + 1 by
//            cp.async into a shared-memory column while tile i is evaluated was measured: long-scoreboard stalls fell
//            from 5.0 to 1.7 per issue, but 33 KB of shared memory per CTA left 23 KB of L1 and the instruction-fetch
//            stalls rose from 1.7 to 4.3 per issue - 0.504 ms against 0.462 ms; profiles/r02_k1p_ncu_summary.md.)
//   scan     every activity id indexes a 16-byte table entry in shared memory and advances the class bit-planes with
//            one integer multiply-add per plane (scan32 below).  Rank space (NKW_RANK): a slot pushes its plane bits
//            only if it holds an event of the pattern, so the planes come out COMPACTED to the filtered list - bit r =
//            r-th relevant event, 32-bit masks, and `position` (EventTs route) / `timestamp` (EventPos route) of an
//            event is its bit index.  Raw space (NKW_RAW): one bit per slot, 64-bit masks, `position` of the EventPos
//            route is the slot.
//   compose  class c = minterm of the planes (one LOP3 each); state k's mask = OR of its classes (uniform branches)
//   walk     NkwWalk: per state one AND of {state mask, above(previous event), predicate windows} and a lowest-set-bit;
//            the first start whose walk completes is the first-largest occurrence (monotone walks)
//   output   fixed staging slots per tile (no atomic on the critical path), the tile's events written as one flat
//            coalesced stream; the placement kernels of detect.cu order them by trace.  A uniform result is staged for
//            gather_uniform_kernel: two words per tile (matched / overflow lanes) instead of per-candidate counts, one
//            packed {pos, rank, act} word and the timestamp per event
// Traces that do not fit (more than 64 slots, or more than 32 relevant events in rank space) go to the overflow list
// and re-run on the staged kernel, launched unconditionally with its work count read from the device.
#include "detect_common.cuh"

namespace siesta {

#ifndef SIESTA_NKP_MIN_CTAS
#define SIESTA_NKP_MIN_CTAS 8
#endif
#ifndef SIESTA_NKP_PREFETCH   // 1: request the next tile's offsets a tile early (six more live registers)
#define SIESTA_NKP_PREFETCH 0
#endif

// The scan.  Every activity id indexes a 16-byte table entry {m, b0, b1, b2} in shared memory (one LDS.128, entry
// n_act = "no event": slots outside the trace) and every plane is advanced with ONE integer multiply-add,
//     plane_p = plane_p * m + b_p,
// which runs on the FMA pipe: shifts and logic ops share the ALU pipe, which takes one warp instruction every two
// cycles, and the walks need that pipe.  Rank space: m = 2 and b_p = plane bit for an activity of the pattern, m = 1 and
// b_p = 0 otherwise - a slot pushes its bits only if it holds a relevant event, so the planes come out compacted to
// the filtered list; the raw relevance mask is advanced as r = 2 r + m (after 32 pushes r + 1 is the mask: each push
// adds m - 1 = the relevance bit plus a constant that sums to 2^32 - 1).  Raw space: m = 2 for every entry.
// The table is kept eight times, entry a of copy c at [a * 8 + c]: lane l reads copy l & 7, so the eight lanes a
// shared-memory wavefront serves (LDS.128: a quarter warp) always sit on eight different bank quads - no bank conflict
// whatever the activity ids are (measured before: 58 M wavefronts for 30 M ideal, the L1 data pipe at 85 % of its peak).
constexpr int LUT_SKEW = 8;
template <int NPL, bool RAW>
__device__ __forceinline__ void scan16(const uint4* __restrict__ lut, const int4 (&v)[4], uint32_t (&pl)[3], uint32_t& racc) {
#pragma unroll
    for (int q = 3; q >= 0; --q) {   // last slot first: bit 0 = first slot / first relevant event
        const int a[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
        for (int i = 3; i >= 0; --i) {
            const uint4 w = lut[a[i] * LUT_SKEW];
            pl[0] = pl[0] * w.x + w.y;
            if (NPL > 1) pl[1] = pl[1] * w.x + w.z;
            if (NPL > 2) pl[2] = pl[2] * w.x + w.w;
            if (!RAW) racc = racc * 2u + w.x;
        }
    }
}

// index of the r-th set bit of x (0-based; r < popc(x)): binary search over popcounts, branch-free
__device__ __forceinline__ int select32(uint32_t x, int r) {
    int pos = 0;
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const int c = __popc((x >> pos) & ((1u << w) - 1u));
        if (r >= c) {
            r -= c;
            pos += w;
        }
    }
    return pos;
}
__device__ __forceinline__ int select64(unsigned long long x, int r) {
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    const int c = __popc(lo);
    return r >= c ? 32 + select32(hi, r - c) : select32(lo, r);
}

template <int NPL, bool RAW, bool MARKOV>
__global__ void __launch_bounds__(NT_MAX, SIESTA_NKP_MIN_CTAS) detect_nkp_kernel(const __grid_constant__ DetectParams P, const __grid_constant__ NkwProgram prog) {
    typedef typename std::conditional<RAW, unsigned long long, uint32_t>::type mask_t;
    typedef unsigned long long u64;
    typedef NkwBits<mask_t> B;
    const int lane = threadIdx.x & 31;
    extern __shared__ uint4 s_lut_all[];   // the table [n_act + 1][LUT_SKEW]
    for (int i = threadIdx.x; i < (P.n_act + 1) * LUT_SKEW; i += blockDim.x) s_lut_all[i] = P.nkp_lut[i / LUT_SKEW];
    __syncthreads();
    const uint4* s_lut = s_lut_all + (lane & (LUT_SKEW - 1));
    const bool evt_pos = (P.flags & SIESTA_F_EVT_POS) != 0;
    const bool all_cols = (P.flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;
    const bool return_all = (P.flags & SIESTA_F_RETURN_ALL) != 0;
    // monotone walks: the first completed start wins; the number of engine matches is only needed for COUNT_MATCHES and for
    // returnAll (one match: it is the selection; more: Occurrence.overlaps decides, on the staged kernel)
    const bool first_only = (P.flags & (SIESTA_F_COUNT_MATCHES | SIESTA_F_RETURN_ALL)) == 0;

    const long long n_work = P.n_work_dev ? (long long)__ldg(P.n_work_dev) : (long long)P.n_work;
    const long long n_tiles = (n_work + 31) / 32;
    const int batch = P.tile_batch;
    // Tiles are handed out by an atomic counter (a CTA that starts late because a collective or a copy holds its SM
    // takes fewer), `batch` consecutive tiles per atomic.  The pipeline needs the next tile's index a whole tile early,
    // so a warp always holds the batch after the current one (next_batch) and requests the one after that (next_batch2)
    // when a batch starts: no atomic is ever waited for.
    long long tile = 0, next_batch = 0, next_batch2 = 0;
    if (lane == 0) {
        tile = (long long)atomicAdd(P.counters + P.tile_slot, (unsigned long long)batch);
        next_batch = (long long)atomicAdd(P.counters + P.tile_slot, (unsigned long long)batch);
    }
    tile = shfl_i64(tile, 0);
    int left = batch;
    unsigned long long acc_occ = 0, acc_ev = 0, acc_emit = 0;  // totals, flushed once per warp

    // the trace of this lane in a tile: candidate index, trace offsets
    auto locate = [&](long long tl, int64_t& ci_, long long& o0_, long long& o1_) {
        const int64_t wi = tl * 32 + lane;
        ci_ = -1;
        o0_ = o1_ = 0;
        if (tl < n_tiles && wi < n_work) {
            ci_ = P.work ? P.work[wi] : wi;
            const int64_t t = P.cand ? P.cand[ci_] : ci_;
            o0_ = P.trace_off[t];
            o1_ = P.trace_off[t + 1];
        }
    };
    int64_t ci;
    long long o0, o1;
    locate(tile, ci, o0, o1);
    while (tile < n_tiles) {
        if (left == batch && lane == 0) next_batch2 = (long long)atomicAdd(P.counters + P.tile_slot, (unsigned long long)batch);
        const long long nxt = left > 1 ? tile + 1 : shfl_i64(next_batch, 0);
#if SIESTA_NKP_PREFETCH
        // the next tile's offsets: requested now, needed when this tile is done
        int64_t nci;
        long long no0, no1;
        locate(nxt, nci, no0, no1);
#endif

        const long long e0 = o0 & ~7LL;
        const int lead = (int)(o0 - e0);
        const long long span = (o1 - o0) + lead;  // slots the trace needs
        bool fits = span <= 64 && ((o1 + 7) & ~7LL) <= P.n_events;
        const long long o1s = fits ? o1 : e0;     // a trace that does not fit is not read here - not even the sector of its first event,
                                                  // which may cross the end of the log (or of a chunk that is still on the host link)
        u64 valid = 0;
        if (fits && o1 > o0) valid = (span == 64 ? ~0ull : ((1ull << (int)span) - 1ull)) & ~((1ull << lead) - 1ull);
        const bool second = __any_sync(0xffffffffu, fits && span > 32);

        // The 64 slots come in quarters of 16 (two 256-bit loads each), last quarter first, double-buffered: the loads of
        // the next quarter are in flight while this one is scanned, and only two quarters (32 registers) are ever live -
        // the kernel fits more warps on an SM than with all 64 slots in registers.
        uint32_t q[3] = {0u, 0u, 0u}, qb[3] = {0u, 0u, 0u}, ra = 0u, rb = 0u;   // RAW: q = slots 0..31, qb = slots 32..63
        {
            int4 A[4], B[4];
            if (second) {
                load_quarter(P, e0 + 48, o1s, A);
                load_quarter(P, e0 + 32, o1s, B);
                scan16<NPL, RAW>(s_lut, A, RAW ? qb : q, rb);
                load_quarter(P, e0 + 16, o1s, A);
                scan16<NPL, RAW>(s_lut, B, RAW ? qb : q, rb);
                load_quarter(P, e0, o1s, B);
                rb += 1u;
            } else {
                load_quarter(P, e0 + 16, o1s, A);
                load_quarter(P, e0, o1s, B);
            }
            scan16<NPL, RAW>(s_lut, A, q, ra);
            scan16<NPL, RAW>(s_lut, B, q, ra);
            ra += 1u;
        }
        mask_t pl[3];
        u64 Rv;   // slots of the trace that hold an event of the pattern
        if constexpr (RAW) {
#pragma unroll
            for (int p = 0; p < 3; ++p) pl[p] = p < NPL ? (((u64)q[p] | ((u64)qb[p] << 32)) & valid) : 0ull;
            Rv = pl[0] | pl[1] | pl[2];
        } else {
            const u64 Rraw = (u64)ra | ((u64)rb << 32);             // includes the neighbours' events in the end sectors
            Rv = Rraw & valid;
            const int n_lead = __popc(ra & ((1u << lead) - 1u));    // relevant events of the previous trace: ranks 0 ..
            const int n_valid = __popcll(Rv);
            if (n_lead + n_valid > 32) fits = false;                // the planes hold 32 ranks
            const uint32_t keep = B::one_shl(n_valid) - 1u;
#pragma unroll
            for (int p = 0; p < 3; ++p) pl[p] = p < NPL ? ((q[p] >> n_lead) & keep) : 0u;
        }
        // state masks.  A state that owns one class (the usual case: classes are state-membership signatures) is the
        // minterm of the planes with host-chosen polarities - three logic ops; otherwise the OR of its classes' minterms
        // (cls_word[c] bit k <=> class c belongs to state k).
        mask_t T[SIESTA_MAX_STATES + 1];
#pragma unroll
        for (int k = 0; k <= SIESTA_MAX_STATES; ++k) {
            T[k] = 0;
            if (k < SIESTA_MAX_STATES && k < prog.n_states) {  // uniform
                if (P.st_single[k]) {
                    mask_t m = ~(mask_t)0;
#pragma unroll
                    for (int p = 0; p < NPL; ++p) m &= pl[p] ^ (mask_t)(long long)(int)P.st_inv[k][p];   // sign-extends to 64 bits
                    T[k] = m;
                } else {
#pragma unroll
                    for (int c = 1; c < (1 << NPL); ++c)
                        if (P.cls_word[c] & (1u << k)) {
                            mask_t m = ~(mask_t)0;
#pragma unroll
                            for (int p = 0; p < NPL; ++p) m &= ((c >> p) & 1) ? pl[p] : ~pl[p];
                            T[k] |= m;
                        }
                }
            }
        }

        int status = ST_NONE;
        unsigned n_emitted = 0;
        mask_t best = 0;
        if (ci >= 0 && o1 > o0) {
            if (!fits) status = ST_OVF;
            else if (Rv) {
                bool hit;
                if constexpr (MARKOV) hit = nkw_eval_markov<mask_t>(prog, T, best, n_emitted);   // all starts at once
                else hit = nkw_eval<mask_t>(prog, T, best, n_emitted, first_only);
                if (hit) status = (return_all && n_emitted > 1) ? ST_OVF : ST_MATCH;
            }
        }

        // ------------------------------------------------------------------ output: fixed staging slots of the tile
        const unsigned my_occ = status == ST_MATCH ? 1u : 0u;
        const unsigned my_ev = status == ST_MATCH ? (unsigned)B::popc(best) : 0u;
        unsigned i1 = my_ev;
        unsigned long long i2 = (status == ST_MATCH) ? n_emitted : 0u;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned y1 = __shfl_up_sync(0xffffffffu, i1, d);
            if (lane >= d) i1 += y1;
        }
        if (!first_only) {   // COUNT_MATCHES / returnAll: the engine's match count is part of the result
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned long long y2 = __shfl_up_sync(0xffffffffu, i2, d);
                if (lane >= d) i2 += y2;
            }
        }
        const unsigned match_bal = __ballot_sync(0xffffffffu, status == ST_MATCH);
        const unsigned n_match = __popc(match_bal);
        acc_occ += n_match;
        acc_ev += i1;     // lane 31 holds the tile totals
        acc_emit += i2;
        const unsigned tot1 = __shfl_sync(0xffffffffu, i1, 31);
        if (lane == 31 && n_match) {   // the tile's share of its block of 256 candidates (8 tiles); one occurrence per match
            unsigned long long* b = P.blk_sums + (tile >> 3);
            atomicAdd(b, (unsigned long long)n_match);
            atomicAdd(b + P.n_blk, (unsigned long long)n_match);
            atomicAdd(b + 2 * P.n_blk, (unsigned long long)i1);
        }
        const long long base1 = P.fix_ev + tile * 32 * P.fix_np;
        const bool uniform = P.tile_words != nullptr;
        if (uniform) {   // the tile's two words replace the per-candidate count and staging place
            const unsigned ovf_bal = __ballot_sync(0xffffffffu, status == ST_OVF);
            if (lane == 0) P.tile_words[tile] = match_bal;
            if (lane == 1) P.tile_words[n_tiles + tile] = ovf_bal;
            if (status == ST_OVF) {
                const unsigned long long at = atomicAdd(P.counters + P.ovf_slot, 1ull);
                P.ovf_list[at] = ci;
            }
        } else if (ci >= 0) {
            P.d_cnt[ci] = my_occ | (my_ev << 16);
            if (status == ST_MATCH) {
                P.d_stage[ci] = base1 + (long long)(i1 - my_ev);
                if (P.fix_occ >= 0) {   // returnAll: the placement reads the event count of every staged occurrence
                    P.d_stage_occ[ci] = P.fix_occ + ci;
                    P.s_occ_nev[P.fix_occ + ci] = (int32_t)my_ev;
                }
            } else if (status == ST_OVF) {
                const unsigned long long at = atomicAdd(P.counters + P.ovf_slot, 1ull);
                P.ovf_list[at] = ci;
            }
        }
        if (tot1 > 0) {
            for (unsigned f0 = 0; f0 < tot1; f0 += 32) {
                const unsigned f = f0 + lane;
                int lo = 0, hi = 31;
#pragma unroll
                for (int it = 0; it < 5; ++it) {
                    const int mid = (lo + hi) >> 1;
                    const unsigned vmid = __shfl_sync(0xffffffffu, i1, mid);
                    if (vmid > f) hi = mid; else lo = mid + 1;
                }
                const int owner = lo & 31;
                const unsigned o_incl = __shfl_sync(0xffffffffu, i1, owner);
                const unsigned o_ev = __shfl_sync(0xffffffffu, my_ev, owner);
                mask_t m;
                if constexpr (RAW) m = (mask_t)shfl_i64((long long)best, owner);
                else m = __shfl_sync(0xffffffffu, best, owner);
                const u64 o_R = (u64)shfl_i64((long long)Rv, owner);
                const long long o_o0 = shfl_i64(o0, owner);
                if (f < tot1) {
                    int k = (int)(f - (o_incl - o_ev));  // k-th event of the owner's occurrence
                    for (; k > 0; --k) m &= m - 1;
                    int j, rank;   // raw slot and index in the filtered list
                    if constexpr (RAW) {
                        j = __ffsll((long long)m) - 1;
                        rank = __popcll(o_R & ((1ull << j) - 1ull));
                    } else {
                        rank = __ffs((int)m) - 1;
                        j = select64(o_R, rank);
                    }
                    const int src = j - (int)(o_o0 & 7);
                    const long long at = base1 + f;
                    if (!all_cols) P.s_ev_pos[at] = src;
                    else {
                        // all three loads leave together: the event's activity and timestamp, and the timestamp of the
                        // first event of the filtered list (Utils.java:51-53: base of the EventTs route's seconds)
                        const long long* tsp = reinterpret_cast<const long long*>(P.ts_ms) + o_o0;
                        const int32_t c_act = __ldg(P.act + o_o0 + src);
                        const long long raw = __ldg(tsp + src);
                        const long long o_t0 = evt_pos ? 0 : __ldg(tsp + (__ffsll((long long)o_R) - 1 - (int)(o_o0 & 7)));
                        if (uniform) {   // src, rank < 64 and act < 255 (at most 64 slots, at most 255 activities)
                            P.s_ev_pos[at] = src | (rank << 8) | (c_act << 16);
                        } else {
                            P.s_ev_pos[at] = src;
                            P.s_ev_rank[at] = rank;
                            P.s_ev_act[at] = c_act;
                        }
                        // SaseEvent.getEventBoth: timestamp * 1000 + minTs (SaseEvent.java:94-106)
                        P.s_ev_ts[at] = evt_pos ? raw : (long long)rel_seconds(raw - o_t0) * 1000 + o_t0;
                    }
                }
            }
        }
        tile = nxt;
        if (--left == 0) {
            left = batch;
            next_batch = next_batch2;
        }
#if SIESTA_NKP_PREFETCH
        ci = nci;
        o0 = no0;
        o1 = no1;
#else
        locate(tile, ci, o0, o1);
#endif
    }
    if (lane == 31) {
        if (acc_occ) {
            atomicAdd(P.counters + 0, acc_occ);
            atomicAdd(P.counters + 6, acc_occ);  // one occurrence per matching trace
        }
        if (acc_ev) atomicAdd(P.counters + 1, acc_ev);
        if (acc_emit) atomicAdd(P.counters + 2, acc_emit);
    }
}

namespace {
template <int NPL, bool RAW, bool MARKOV>
int launch_one(const Ctx* ctx, cudaStream_t stream, DetectParams P, const NkwProgram& prog) {
    auto kern = detect_nkp_kernel<NPL, RAW, MARKOV>;
    const size_t smem = (size_t)(P.n_act + 1) * LUT_SKEW * sizeof(uint4);
    int per_sm = 0;
    SIESTA_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, smem));
    if (per_sm < 1) per_sm = 1;
    if (const char* env = std::getenv("SIESTA_K1_CTAS_PER_SM")) {  // tuning aid: cap on resident CTAs per SM
        const int v = std::atoi(env);
        if (v >= 1 && v < per_sm) per_sm = v;
    }
    if (const char* env = std::getenv("SIESTA_NKP_CARVEOUT")) {  // tuning aid: shared-memory carveout in percent
        const int v = std::atoi(env);
        if (v >= 0 && v <= 100) SIESTA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    }
    const int64_t n_tiles = (P.n_work + 31) / 32;
    const int64_t ctas_needed = (n_tiles + NT / 32 - 1) / (NT / 32);
    int grid = (int)std::min<int64_t>(ctas_needed, (int64_t)ctx->sm_count * per_sm);
    if (grid < 1) grid = 1;
    // a batch of tiles per atomic once every warp has many batches to take (the tail stays balanced)
    const int64_t per_warp = n_tiles / ((int64_t)grid * (NT / 32));
    P.tile_batch = per_warp >= 64 ? 4 : (per_warp >= 16 ? 2 : 1);
    if (const char* env = std::getenv("SIESTA_NKP_TILE_BATCH")) {
        const int v = std::atoi(env);
        if (v >= 1 && v <= 64) P.tile_batch = v;
    }
    kern<<<grid, NT, smem, stream>>>(P, prog);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}
}  // namespace

int launch_nkp(const Ctx* ctx, cudaStream_t stream, const DetectParams& P, const NkwProgram& prog, int space) {
    const bool raw = space == NKW_RAW;
    const bool markov = prog.markov && std::getenv("SIESTA_NKP_NO_MARKOV") == nullptr;
#define SIESTA_NKP_GO(NPL)                                                                                              \
    (raw ? (markov ? launch_one<NPL, true, true>(ctx, stream, P, prog) : launch_one<NPL, true, false>(ctx, stream, P, prog))   \
         : (markov ? launch_one<NPL, false, true>(ctx, stream, P, prog) : launch_one<NPL, false, false>(ctx, stream, P, prog)))
    if (P.n_planes == 1) return SIESTA_NKP_GO(1);
    if (P.n_planes == 2) return SIESTA_NKP_GO(2);
    return SIESTA_NKP_GO(3);
#undef SIESTA_NKP_GO
}

}  // namespace siesta
