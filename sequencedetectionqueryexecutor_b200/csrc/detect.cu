// detect.cu — kernel K1: per-trace pattern verification over a CSR event log (sm_100a).
//
// Replaces SaseConnector.evaluate + Occurrences.clearOccurrences
// (J/SaseConnection/SaseConnector.java:48-76, J/model/Occurrences.java:58-89).
//
// Launch shape: persistent CTAs of NT = 128 threads (grid = SMs x resident CTAs); every WARP owns a tile of 32 traces
// from start to finish, one lane per trace, no block-level barrier; tiles are handed out by an atomic counter.
//   detect_kernel (staged, every NFA class)
//     phase A  each lane streams its own trace in 32-byte sectors, tests the activity ids against the pattern's class
//              bit-planes in registers and appends the surviving events (the reference's Trace.clearTrace /
//              Utils.transformToSaseEvents) to its lane-transposed shared-memory column; timestamps (int64 ms) travel by
//              cp.async, for surviving events only
//     phase B  one lane per trace: closed-form evaluators (detect_fast.cuh: classes NK and FK2) or the run-list engine
//              (detect_engine.cuh)
//     phase C  warp scan of the output sizes, one reservation per tile, the tile's events written as one flat stream
//   detect_nkp_kernel (K1-P: class NK, first-largest occurrence, no relative seconds)
//              no shared memory: class planes of the trace's 64 raw position slots in registers, one mask per NFA
//              state, greedy walks on the masks, fixed staging slots (no atomic on the critical path)
//   count_blocks / scan_chunks / scan_top / gather
//              order the staged occurrences by trace index (dense per-candidate counts + device scans), so the
//              result is deterministic
// A request is two host-side halves (detect_device_begin_impl: kernels enqueued, nothing waited for;
// detect_device_finish_impl: sizes, result allocation, placement), exposed as siesta_detect_device_begin / _finish
// and, in one call, siesta_detect_device.
#include <algorithm>
#include <cstdio>
#include <type_traits>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "detect_common.cuh"

namespace siesta {

// Shared memory of one warp (all arrays lane-transposed: element i of lane l at [i * 32 + l]).
template <int W, int R, int NF, bool SMEM_RUNS>
struct WarpSmem {
    static constexpr int NE = ROWS_OF(W);
    static constexpr size_t famvv_off = 0;
    static constexpr size_t famvv_bytes = SMEM_RUNS ? sizeof(unsigned long long) * NF * 32 : 0;
    static constexpr size_t rmask_off = famvv_off + famvv_bytes;
    static constexpr size_t rmask_bytes = SMEM_RUNS ? sizeof(typename MaskOps<W>::T) * R * 32 : 0;
    // per event, while the trace is scanned: class | in-trace index << 3; afterwards: the activity id
    // (16 bits in the narrow configuration: traces longer than 8192 events go to the wide one)
    typedef typename std::conditional<W == 1, uint16_t, uint32_t>::type small_t;
    static constexpr size_t small_off = rmask_off + rmask_bytes;
    static constexpr size_t small_bytes = sizeof(small_t) * NE * 32;
    static constexpr size_t rmeta_off = (small_off + small_bytes + 15) & ~(size_t)15;
    static constexpr size_t rmeta_bytes = SMEM_RUNS ? sizeof(uint32_t) * R * 32 : 0;
    static constexpr size_t bytes_off = rmeta_off + rmeta_bytes;                 // rfam, fmin, fmin2, fcnt
    static constexpr size_t bytes_bytes = SMEM_RUNS ? (size_t)(R + 3 * NF) * 32 : 0;
    // one 8-byte slot per event: first the raw int64 timestamp (cp.async target), then {relative seconds, lut word | index << 16}
    static constexpr size_t slot_off = (bytes_off + bytes_bytes + 15) & ~(size_t)15;
    static constexpr size_t slot_bytes = sizeof(unsigned long long) * NE * 32;
    static constexpr size_t aux_off = slot_off + slot_bytes;
    static constexpr size_t aux_bytes = sizeof(typename MaskOps<W>::T) * NE * 32;   // NK + returnAll: one mask per start
    static __host__ __device__ constexpr size_t total(bool needs_aux) { return aux_off + (needs_aux ? aux_bytes : 0); }
};

// One warp owns a tile of 32 traces from start to finish: no block-level barrier anywhere.
// MODE: FAST_NONE = run-list engine, FAST_NK / FAST_FK2 = closed-form evaluators (detect_fast.cuh).
template <int W, int R, int NF, bool SMEM_RUNS, int MODE>
__global__ void __launch_bounds__(NT_MAX, (W == 1 && MODE != FAST_NONE) ? 5 : 4) detect_kernel(const __grid_constant__ DetectParams P, const __grid_constant__ DevNfa nfa) {
    typedef MaskOps<W> MO;
    typedef typename MO::T mask_t;
    typedef WarpSmem<W, R, NF, SMEM_RUNS> L;
    constexpr int NE = ROWS_OF(W);  // pattern-relevant events a trace may hold in this configuration

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool evt_pos = (P.flags & SIESTA_F_EVT_POS) != 0;
    const bool return_all = (P.flags & SIESTA_F_RETURN_ALL) != 0;
    const bool needs_aux = MODE == FAST_NK && return_all;
    unsigned char* wbase = smem_raw + (size_t)warp * L::total(needs_aux);
    typedef typename L::small_t small_t;
    constexpr unsigned ACT_NONE = W == 1 ? 0xFFFFu : 0xFFFFFFFFu;  // the activity id does not fit small_t: re-read it from the log
    constexpr long long MAX_LEN = W == 1 ? 8192 : 65536;  // the in-trace index must fit small_t next to the class (and 16 bits of the word)
    small_t* s_small = reinterpret_cast<small_t*>(wbase + L::small_off);                      // [NE][32]
    unsigned long long* s_slot = reinterpret_cast<unsigned long long*>(wbase + L::slot_off);  // [NE][32]
    const uint32_t* s_w32 = reinterpret_cast<const uint32_t*>(s_slot);  // slot j of lane l: words [(j * 32 + l) * 2 + {0: seconds, 1: word}]

    const bool all_cols = (P.flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;
    const bool prune = (P.flags & SIESTA_F_LITERAL_RUNS) == 0;
    const bool dedup = prune && !return_all && (P.flags & SIESTA_F_COUNT_MATCHES) == 0;

    const long long n_work = P.n_work_dev ? (long long)__ldg(P.n_work_dev) : (long long)P.n_work;
    const long long n_tiles = (n_work + 31) / 32;
    // Tiles are handed out by an atomic counter, not by a static stride: when another kernel (an NCCL all-gather of the
    // previous request's results, a copy) holds some SMs, the CTAs that start late simply take fewer tiles.  The next
    // tile is requested at the top of the loop so that the atomic's latency hides behind the current tile.
    long long tile = 0;
    if (lane == 0) tile = (long long)atomicAdd(P.counters + P.tile_slot, 1ull);
    tile = shfl_i64(tile, 0);
    // Totals that nobody waits for are summed per warp (lane 31) and flushed once after the last tile: all counters of
    // a launch share one 128-byte line, and same-line atomics are served one at a time by the L2.
    unsigned long long acc_occ = 0, acc_emit = 0, acc_match = 0;
    while (tile < n_tiles) {
        long long next_tile = 0;
        if (lane == 0) next_tile = (long long)atomicAdd(P.counters + P.tile_slot, 1ull);
        // ------------------------------------------------------------------ phase A: filter + compact, one lane per trace
        // Each lane streams its own trace in 32-byte sectors (two 128-bit loads = 8 activity ids), tests the ids against
        // the pattern's type set in registers, and appends the surviving events to its lane-transposed shared-memory
        // column (the reference's Trace.clearTrace / Utils.transformToSaseEvents).  Timestamps (int64 ms) are loaded
        // only for surviving events, after the scan, as independent loads.
#ifdef SIESTA_PHASE_TIMING
        long long tA = clock64();
#endif
        const int64_t wi = tile * 32 + lane;   // index into the work list
        int64_t ci = -1, t = -1;               // candidate index, trace index
        long long o0 = 0, o1 = 0;
        if (wi < n_work) {
            ci = P.work ? P.work[wi] : wi;
            t = P.cand ? P.cand[ci] : ci;
            o0 = P.trace_off[t];
            o1 = P.trace_off[t + 1];
        }
        int cnt = 0;
        const long long* tsp = reinterpret_cast<const long long*>(P.ts_ms) + o0;
        int4 v[8];
        load_sectors(P, o0 & ~7LL, o0, o1, v);
        for (long long e = o0 & ~7LL; e < o1; e += 32) {  // lanes whose trace has ended leave the loop
            int4 nv[8];
            if (e + 32 < o1) load_sectors(P, e + 32, o0, o1, nv);  // the next 32 events are in flight while these are tested
            // class bit-planes of the 32 events (bit i = event e + i); pend = events that belong to the pattern
            uint32_t pl[3] = {0u, 0u, 0u};
            if (P.alpha_mode == 0) {
                if (P.n_planes == 1) scan_block<1, false>(P, v, pl);
                else if (P.n_planes == 2) scan_block<2, false>(P, v, pl);
                else scan_block<3, false>(P, v, pl);
            } else if (P.alpha_mode == 1) {
                if (P.n_planes == 1) scan_block<1, true>(P, v, pl);
                else if (P.n_planes == 2) scan_block<2, true>(P, v, pl);
                else scan_block<3, true>(P, v, pl);
            } else {
#pragma unroll
                for (int q = 7; q >= 0; --q) {
                    const int a[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
                    for (int i = 3; i >= 0; --i) {
                        const bool rel = ((unsigned)a[i] < (unsigned)P.n_act) && __ldg(P.lut + a[i]) != 0;
                        pl[0] = (pl[0] << 1) | (rel ? 1u : 0u);
                    }
                }
            }
            uint32_t pend = pl[0] | pl[1] | pl[2];
            // events of the neighbouring traces that share the first / last sector
            if (e < o0) pend &= ~((1u << (int)(o0 - e)) - 1u);
            if (o1 - e < 32) pend &= (1u << (int)(o1 - e)) - 1u;
            while (pend) {
                const int j = __ffs(pend) - 1;
                pend &= pend - 1;
                if (cnt < NE) {
                    const long long src = e + j - o0;
                    const uint32_t cls = ((pl[0] >> j) & 1u) | (((pl[1] >> j) & 1u) << 1) | (((pl[2] >> j) & 1u) << 2);
                    s_small[cnt * 32 + lane] = (small_t)(cls | ((uint32_t)src << 3));
                    // the raw timestamp of a surviving event goes straight to its shared-memory slot (no register, no stall)
                    if (P.needs_ts) cp_async8(s_slot + cnt * 32 + lane, tsp + src);
                }
                ++cnt;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = nv[q];
        }
        if (o1 - o0 > MAX_LEN) cnt = NE + 1;  // in-trace index does not fit the packed word: overflow path
        const int my_cnt = cnt;
        cp_async_wait_all();
        // second pass over the survivors only: activity -> state-mask word, timestamp -> relative seconds
        long long t0ms = 0;  // first event of the filtered list (Utils.java:51-53)
        if (my_cnt > 0 && my_cnt <= NE) {
            if (P.needs_ts) t0ms = (long long)s_slot[lane];
            else if (all_cols && !evt_pos) t0ms = __ldg(tsp + (s_small[lane] >> 3));
#pragma unroll 4
            for (int r = 0; r < my_cnt; ++r) {
                const uint32_t cw = s_small[r * 32 + lane];
                const uint32_t src = cw >> 3;
                int a;
                uint32_t m;
                if (P.alpha_mode == 2) {  // general alphabet: re-read the activity (L2 hit) and look its word up
                    a = __ldg(P.act + o0 + src);
                    m = (uint32_t)__ldg(P.lut + a);
                } else {
                    a = P.cls_act[cw & 7u];
                    m = (uint32_t)P.cls_word[cw & 7u];
                }
                int rel = 0;
                if (P.needs_ts) rel = rel_seconds((long long)s_slot[r * 32 + lane] - t0ms);
                s_slot[r * 32 + lane] = (unsigned long long)(uint32_t)rel | ((unsigned long long)(m | (src << 16)) << 32);
                s_small[r * 32 + lane] = (small_t)((unsigned)a < ACT_NONE ? (unsigned)a : ACT_NONE);
            }
        }
        __syncwarp();

        // ------------------------------------------------------------------ phase B: one lane per trace
#ifdef SIESTA_PHASE_TIMING
        long long tB = clock64();
#endif
        int status = ST_NONE;
        unsigned n_emitted = 0;
        int nsel = 0;
        mask_t sel_local[(MODE == FAST_FK2 || MODE == FAST_NP1) ? 1 : NE];
        if (ci >= 0 && my_cnt > 0) {
            if (my_cnt > NE) {
                status = ST_OVF;
            } else {
                TraceEvents ev{s_w32 + 2 * lane + 1, P.needs_ts ? reinterpret_cast<const int32_t*>(s_w32) + 2 * lane : nullptr,
                               64, my_cnt, evt_pos, 64};
                if constexpr (MODE == FAST_FK2) {
                    mask_t m = 0;
                    if (fk2_eval<W>(nfa, ev, m)) {
                        status = ST_MATCH;
                        sel_local[0] = m;
                        nsel = 1;
                    }
                } else if constexpr (MODE == FAST_NP1) {
                    NkMasks<W> nkm;
                    nkm.init();
                    for (int j = 0; j < ev.n; ++j) nkm.on_event(j, ev.word(j));
                    const bool count = (P.flags & (SIESTA_F_RETURN_ALL | SIESTA_F_COUNT_MATCHES)) != 0;
                    if (nfa.need_vv ? np1p_eval<W>(nfa, ev, nkm.T, sel_local[0], n_emitted) : np1_eval<W>(nfa, nkm.T, count, sel_local[0], n_emitted)) {
                        status = ST_MATCH;
                        nsel = 1;
                    }
                } else if constexpr (MODE == FAST_NK) {
                    mask_t* aux = reinterpret_cast<mask_t*>(wbase + L::aux_off) + lane;
                    NkMasks<W> nkm;
                    nkm.init();
                    for (int j = 0; j < ev.n; ++j) nkm.on_event(j, ev.word(j));
                    if (nk_eval<W>(nfa, ev, nkm.T, return_all, evt_pos, aux, 32, sel_local, nsel, n_emitted)) status = ST_MATCH;
                } else {
                    auto body = [&](auto& eng) {
                        BestEmit<W> be;
                        eng.run(be, prune, dedup);
                        if (eng.ovf) status = ST_OVF;
                        else if (eng.err) status = ST_ERR;
                        else if (be.n > 0) {
                            status = ST_MATCH;
                            n_emitted = be.n;
                            sel_local[0] = be.best;
                            nsel = 1;
                            if (return_all && be.n > 1) {
                                GreedyEmit<W, NE> ge(ev, be.best, evt_pos);
                                eng.run(ge, prune, false);
                                if (ge.ovf || eng.ovf) status = ST_OVF;
                                else {
                                    nsel = ge.nsel;
                                    for (int o = 1; o < nsel; ++o) sel_local[o] = ge.sel[o];
                                }
                            }
                        }
                    };
                    if constexpr (SMEM_RUNS) {
                        uint8_t* bytes = wbase + L::bytes_off + lane;
                        RunStore<W, R, NF, 32> store{reinterpret_cast<mask_t*>(wbase + L::rmask_off) + lane,
                                                     reinterpret_cast<uint32_t*>(wbase + L::rmeta_off) + lane,
                                                     bytes,
                                                     reinterpret_cast<unsigned long long*>(wbase + L::famvv_off) + lane,
                                                     bytes + (size_t)R * 32, bytes + (size_t)(R + NF) * 32, bytes + (size_t)(R + 2 * NF) * 32};
                        RunEngine<RunStore<W, R, NF, 32>> eng(nfa, ev, store);
                        body(eng);
                    } else {
                        RunArrays<W, R, NF> arrays;
                        RunEngine<RunStore<W, R, NF, 1>> eng(nfa, ev, arrays.store());
                        body(eng);
                    }
                }
            }
        }

        // ------------------------------------------------------------------ phase C: reserve staging space per warp, write
#ifdef SIESTA_PHASE_TIMING
        __syncwarp();
        long long tC = clock64();
#endif
        unsigned my_occ = 0, my_ev = 0;
        if (status == ST_MATCH) {
            my_occ = (unsigned)nsel;
            for (int o = 0; o < nsel; ++o) my_ev += MO::popc(sel_local[o]);
        }
        unsigned i0 = my_occ, i1 = my_ev;
        unsigned long long i2 = (status == ST_MATCH) ? n_emitted : 0u;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned y0 = __shfl_up_sync(0xffffffffu, i0, d), y1 = __shfl_up_sync(0xffffffffu, i1, d);
            const unsigned long long y2 = __shfl_up_sync(0xffffffffu, i2, d);
            if (lane >= d) { i0 += y0; i1 += y1; i2 += y2; }
        }
        const unsigned n_match = __popc(__ballot_sync(0xffffffffu, status == ST_MATCH));
        unsigned long long base0 = 0, base1 = 0;
        if (lane == 31) {
            // with one occurrence per trace the occurrence is staged at the candidate's own index: one reservation per tile
            if (return_all) { if (i0) base0 = atomicAdd(P.counters + 0, (unsigned long long)i0); }
            else acc_occ += i0;
            if (i1) base1 = atomicAdd(P.counters + 1, (unsigned long long)i1);
            acc_emit += i2;
            acc_match += n_match;
        }
        const unsigned tot0 = __shfl_sync(0xffffffffu, i0, 31), tot1 = __shfl_sync(0xffffffffu, i1, 31);
        if (P.work == nullptr) {          // a tile of 32 consecutive candidates: one reduction per tile
            if (lane == 31 && n_match) {
                unsigned long long* b = P.blk_sums + (tile >> 3);
                atomicAdd(b, (unsigned long long)n_match);
                atomicAdd(b + P.n_blk, (unsigned long long)i0);
                atomicAdd(b + 2 * P.n_blk, (unsigned long long)i1);
            }
        } else if (status == ST_MATCH) {  // a re-run list: the candidates come from anywhere
            unsigned long long* b = P.blk_sums + (ci >> 8);
            atomicAdd(b, 1ull);
            atomicAdd(b + P.n_blk, (unsigned long long)my_occ);
            atomicAdd(b + 2 * P.n_blk, (unsigned long long)my_ev);
        }
        base0 = __shfl_sync(0xffffffffu, base0, 31);
        base1 = __shfl_sync(0xffffffffu, base1, 31);
        const long long occ_at = return_all ? (long long)(base0 + i0 - my_occ) : (long long)ci;
        const long long ev_at = (long long)(base1 + i1 - my_ev);
        const bool stage_ok = (!return_all || (long long)(base0 + tot0) <= P.cap_occ) && (long long)(base1 + tot1) <= P.cap_ev;
        if (!stage_ok && lane == 0) atomicAdd(P.counters + 5, 1ull);

        if (ci >= 0) {
            if (status == ST_MATCH) {
                P.d_cnt[ci] = my_occ | (my_ev << 16);
                P.d_stage[ci] = ev_at;
                if (return_all) P.d_stage_occ[ci] = occ_at;
            } else {
                P.d_cnt[ci] = 0;
                if (status == ST_ERR) P.err_list[atomicAdd(P.counters + 3, 1ull)] = t;
                else if (status == ST_OVF) {
                    const unsigned long long at = atomicAdd(P.counters + P.ovf_slot, 1ull);
                    if (P.ovf_list && (P.ovf_cap == 0 || (long long)at < P.ovf_cap)) P.ovf_list[at] = ci;
                }
            }
        }
        if (stage_ok && tot1 > 0) {
            if (!return_all) {
                // One occurrence per trace: the warp writes the tile's events as one flat, coalesced stream.  Flat slot
                // f belongs to the lane whose inclusive event count first exceeds f (binary search over shuffles); the
                // k-th set bit of that lane's occurrence mask names the event; activity and timestamp are re-read
                // from the log by 32 lanes at once (one memory latency per 32 events instead of one per event).
                const mask_t my_mask = status == ST_MATCH ? sel_local[0] : (mask_t)0;
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
                    if constexpr (W == 1) m = __shfl_sync(0xffffffffu, my_mask, owner);
                    else m = (mask_t)shfl_i64((long long)my_mask, owner);
                    const long long o_o0 = shfl_i64(o0, owner);
                    const long long o_t0 = shfl_i64(t0ms, owner);
                    if (f < tot1) {
                        int k = (int)(f - (o_incl - o_ev));  // k-th event of the owner's occurrence
                        for (; k > 0; --k) m &= m - 1;
                        const int j = MO::lo(m);
                        const unsigned long long slot = s_slot[j * 32 + owner];  // {relative seconds, lut word | index << 16}
                        const int src = (int)(slot >> 48);
                        const long long at = (long long)base1 + f;
                        P.s_ev_pos[at] = src;
                        if (all_cols) {
                            const uint32_t sa = s_small[j * 32 + owner];
                            P.s_ev_rank[at] = j;
                            P.s_ev_act[at] = sa != ACT_NONE ? (int32_t)sa : __ldg(P.act + o_o0 + src);
                            // SaseEvent.getEventBoth: timestamp * 1000 + minTs (SaseEvent.java:94-106)
                            long long out_ts;
                            if (P.needs_ts) out_ts = (long long)(int32_t)(uint32_t)slot * 1000 + o_t0;
                            else {
                                const long long raw = __ldg(reinterpret_cast<const long long*>(P.ts_ms) + o_o0 + src);
                                out_ts = evt_pos ? raw : (long long)rel_seconds(raw - o_t0) * 1000 + o_t0;
                            }
                            P.s_ev_ts[at] = out_ts;
                        }
                    }
                }
            } else if (status == ST_MATCH) {
                long long e = ev_at;
                for (int o = 0; o < nsel; ++o) {
                    mask_t m = sel_local[o];
                    P.s_occ_nev[occ_at + o] = MO::popc(m);
                    while (m) {
                        const int j = MO::lo(m);
                        m &= m - 1;
                        const unsigned long long slot = s_slot[j * 32 + lane];  // {relative seconds, lut word | index << 16}
                        const int src = (int)(slot >> 48);
                        P.s_ev_pos[e] = src;
                        if (all_cols) {
                            const uint32_t sa = s_small[j * 32 + lane];
                            P.s_ev_rank[e] = j;
                            P.s_ev_act[e] = sa != ACT_NONE ? (int32_t)sa : __ldg(P.act + o0 + src);
                            // SaseEvent.getEventBoth: timestamp * 1000 + minTs (SaseEvent.java:94-106)
                            long long out_ts;
                            if (P.needs_ts) out_ts = (long long)(int32_t)(uint32_t)slot * 1000 + t0ms;
                            else {
                                const long long raw = __ldg(reinterpret_cast<const long long*>(P.ts_ms) + o0 + src);
                                out_ts = evt_pos ? raw : (long long)rel_seconds(raw - t0ms) * 1000 + t0ms;
                            }
                            P.s_ev_ts[e] = out_ts;
                        }
                        ++e;
                    }
                }
            }
        }
#ifdef SIESTA_PHASE_TIMING
        {
            long long tD = clock64();
            if (lane == 0) {
                atomicAdd(P.counters + 8, (unsigned long long)(tB - tA));
                atomicAdd(P.counters + 9, (unsigned long long)(tC - tB));
                atomicAdd(P.counters + 10, (unsigned long long)(tD - tC));
            }
        }
#endif
        __syncwarp();  // the warp's shared-memory slot is reused by its next tile
        tile = shfl_i64(next_tile, 0);
    }
    if (lane == 31) {
        if (acc_occ) atomicAdd(P.counters + 0, acc_occ);
        if (acc_emit) atomicAdd(P.counters + 2, acc_emit);
        if (acc_match) atomicAdd(P.counters + 6, acc_match);
    }
}

// ---------------------------------------------------------------------------------- K1-L: class NK on traces of any length
// The traces the wide launch could not hold (more than 64 pattern-relevant events, more than 65 536 events) re-run here when
// the NFA has no Kleene state: one warp per trace, no masks.  Phase A compacts the trace's relevant events into plain arrays
// (state word, position, relative seconds) carved from a bump-allocated pool; phase B walks every start forward through
// that list, lanes = starts (nk_long_walk, detect_fast.cuh); phase C selects as Occurrences.clearOccurrences does - the
// smallest (completion, start), then, for returnAll, the later runs in emission order that overlap nothing chosen - and
// stages the events in a region of its own.  A trace that does not fit the pool, the staging region or the 16-bit
// per-trace counts of the placement goes to the final list of unsupported traces.
struct LongParams {
    const int64_t* work;                     // candidate indices (the wide launch's overflow list)
    const unsigned long long* n_work_dev;
    int64_t work_cap;
    char* pool;
    unsigned long long pool_bytes;
    int64_t ev_base, ev_cap;                 // staging region of this kernel inside the s_ev_* arrays
    int64_t occ_base, occ_cap;               // ... inside s_occ_nev (returnAll)
    int64_t* unsup;                          // final list of unsupported traces (candidate indices)
    int64_t unsup_cap;
    int32_t n_positive;
    // counters: 14 final unsupported, 19 next work item, 20 pool cursor, 21 staged events, 22 staged occurrences
};

__global__ void __launch_bounds__(128) detect_long_kernel(const __grid_constant__ DetectParams P, const __grid_constant__ LongParams Q,
                                                          const __grid_constant__ DevNfa nfa) {
    const int lane = threadIdx.x & 31;
    const bool evt_pos = (P.flags & SIESTA_F_EVT_POS) != 0;
    const bool return_all = (P.flags & SIESTA_F_RETURN_ALL) != 0;
    const bool all_cols = (P.flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;
    const int np = Q.n_positive;
    long long n_work = (long long)__ldg(Q.n_work_dev);
    if (n_work > Q.work_cap) n_work = Q.work_cap;   // (the host fails the request beyond the cap)
    for (;;) {
        long long w = 0;
        if (lane == 0) w = (long long)atomicAdd(P.counters + 19, 1ull);
        w = shfl_i64(w, 0);
        if (w >= n_work) break;
        const int64_t ci = Q.work[w];
        const int64_t t = P.cand ? P.cand[ci] : ci;
        const long long o0 = P.trace_off[t], o1 = P.trace_off[t + 1];
        const long long len = o1 - o0;
        bool ok = len <= 0x7fffffffll;
        // ---- pool: word u16[len] | pos i32[len] | sec i32[len] | rec_c i32[len] | rec_e i32[len * np] | sel i32[len]
        const unsigned long long need = ((unsigned long long)len * (2 + 4 + 4 + 4 + 4 * (unsigned)np + 4) + 255) & ~255ull;
        unsigned long long at = 0;
        if (lane == 0 && ok) at = atomicAdd(P.counters + 20, need);
        at = (unsigned long long)shfl_i64((long long)at, 0);
        ok = ok && at + need <= Q.pool_bytes;
        int n_rel = 0, nsel = 0;
        unsigned n_emitted = 0;
        long long t0ms = 0;
        int32_t *pos = nullptr, *sec = nullptr, *rec_c = nullptr, *rec_e = nullptr, *sel = nullptr;
        uint16_t* word = nullptr;
        if (ok) {
            char* base = Q.pool + at;
            pos = reinterpret_cast<int32_t*>(base);
            sec = pos + len;
            rec_c = sec + len;
            rec_e = rec_c + len;
            sel = rec_e + len * np;
            word = reinterpret_cast<uint16_t*>(sel + len);
            // ---- phase A: compact the relevant events (lanes = events, coalesced)
            bool have_t0 = false;
            for (long long e0 = 0; e0 < len; e0 += 32) {
                const long long e = e0 + lane;
                uint32_t wd = 0;
                long long raw = 0;
                if (e < len) {
                    const int a = __ldg(P.act + o0 + e);
                    if ((unsigned)a < (unsigned)P.n_act) wd = (uint32_t)__ldg(P.lut + a) & 0xFFu;
                    if (wd && (P.needs_ts || (all_cols && !evt_pos))) raw = __ldg(reinterpret_cast<const long long*>(P.ts_ms) + o0 + e);
                }
                const unsigned m = __ballot_sync(0xffffffffu, wd != 0);
                if (!have_t0 && m) {   // first event of the filtered list (Utils.java:51-53)
                    t0ms = shfl_i64(raw, __ffs((int)m) - 1);
                    have_t0 = true;
                }
                if (wd) {
                    const int r = n_rel + __popc(m & ((1u << lane) - 1u));
                    word[r] = (uint16_t)wd;
                    pos[r] = (int32_t)e;
                    sec[r] = P.needs_ts ? rel_seconds(raw - t0ms) : 0;
                    rec_c[r] = -1;
                }
                n_rel += __popc(m);
            }
            __syncwarp();
            // ---- phase B: every start's run, lanes = starts
            LongEvents ev{n_rel, word, pos, P.needs_ts ? sec : nullptr, evt_pos};
            int best_c = 0x7fffffff, best_s = 0x7fffffff;
            for (int j0 = 0; j0 < n_rel; j0 += 32) {
                const int j = j0 + lane;
                if (j < n_rel && (word[j] & 1u)) {
                    int o[SIESTA_MAX_STATES];
                    const int k = nk_long_walk(nfa, ev, j, o);
                    if (k) {
                        for (int i = 0; i < k; ++i) rec_e[(long long)j * np + i] = o[i];
                        rec_c[j] = o[k - 1];
                        ++n_emitted;
                        if (o[k - 1] < best_c || (o[k - 1] == best_c && j < best_s)) { best_c = o[k - 1]; best_s = j; }
                    }
                }
            }
#pragma unroll
            for (int d = 16; d; d >>= 1) {
                n_emitted += __shfl_xor_sync(0xffffffffu, n_emitted, d);
                const int oc = __shfl_xor_sync(0xffffffffu, best_c, d), os = __shfl_xor_sync(0xffffffffu, best_s, d);
                if (oc < best_c || (oc == best_c && os < best_s)) { best_c = oc; best_s = os; }
            }
            __syncwarp();
            // ---- phase C: selection (Occurrences.java:58-89)
            if (n_emitted) {
                if (lane == 0) { sel[0] = best_s; rec_c[best_s] = -2 - best_c; }   // taken: completion kept as -2 - c
                nsel = 1;
                __syncwarp();
                if (return_all && n_emitted > 1) {
                    const bool by_pos = evt_pos;
                    for (unsigned round = 1; round < n_emitted; ++round) {
                        // the next run in emission order: smallest (completion, start) among those not looked at yet
                        int mc = 0x7fffffff, ms = 0x7fffffff;
                        for (int j = lane; j < n_rel; j += 32) {
                            const int c = rec_c[j];
                            if (c >= 0 && (c < mc || (c == mc && j < ms))) { mc = c; ms = j; }
                        }
#pragma unroll
                        for (int d = 16; d; d >>= 1) {
                            const int oc = __shfl_xor_sync(0xffffffffu, mc, d), os = __shfl_xor_sync(0xffffffffu, ms, d);
                            if (oc < mc || (oc == mc && os < ms)) { mc = oc; ms = os; }
                        }
                        bool ov = false;   // against every chosen run, lanes = chosen runs
                        for (int q = lane; q < nsel; q += 32) {
                            const int bs = sel[q];
                            const int bl = -2 - rec_c[bs];
                            ov = ov || nk_long_overlaps(ev, by_pos, ms, mc, bs, bl);
                        }
                        ov = __any_sync(0xffffffffu, ov);
                        if (lane == 0) {
                            if (!ov) { sel[nsel] = ms; rec_c[ms] = -2 - mc; }
                            else rec_c[ms] = -1;                                   // looked at, not chosen
                        }
                        if (!ov) ++nsel;
                        __syncwarp();
                    }
                }
            }
        }
        // ---- output
        const long long n_ev = (long long)nsel * np;
        long long ev_at = 0, occ_at = 0;
        if (ok && nsel) {
            ok = nsel <= 0xFFFF && n_ev <= 0xFFFF;   // the placement packs both counts into 16 bits
            if (ok && lane == 0) {
                ev_at = (long long)atomicAdd(P.counters + 21, (unsigned long long)n_ev);
                if (return_all) occ_at = (long long)atomicAdd(P.counters + 22, (unsigned long long)nsel);
            }
            ev_at = shfl_i64(ev_at, 0);
            occ_at = shfl_i64(occ_at, 0);
            ok = ok && ev_at + n_ev <= Q.ev_cap && (!return_all || occ_at + nsel <= Q.occ_cap);
        }
        if (!ok) {
            if (lane == 0) {
                P.d_cnt[ci] = 0;
                const unsigned long long u = atomicAdd(P.counters + 14, 1ull);
                if ((long long)u < Q.unsup_cap) Q.unsup[u] = ci;
            }
            continue;
        }
        if (lane == 0) {
            P.d_cnt[ci] = (uint32_t)nsel | ((uint32_t)n_ev << 16);
            if (nsel) {
                P.d_stage[ci] = Q.ev_base + ev_at;
                if (return_all) P.d_stage_occ[ci] = Q.occ_base + occ_at;
                unsigned long long* b = P.blk_sums + (ci >> 8);
                atomicAdd(b, 1ull);
                atomicAdd(b + P.n_blk, (unsigned long long)nsel);
                atomicAdd(b + 2 * P.n_blk, (unsigned long long)n_ev);
                atomicAdd(P.counters + 0, (unsigned long long)nsel);
                atomicAdd(P.counters + 1, (unsigned long long)n_ev);
                atomicAdd(P.counters + 6, 1ull);
            }
            if (n_emitted) atomicAdd(P.counters + 2, (unsigned long long)n_emitted);
        }
        for (long long f = lane; f < n_ev; f += 32) {
            const int o = (int)(f / np), i = (int)(f % np);
            const int j = rec_e[(long long)sel[o] * np + i];
            const int src = pos[j];
            const long long dst = Q.ev_base + ev_at + f;
            P.s_ev_pos[dst] = src;
            if (all_cols) {
                P.s_ev_rank[dst] = j;
                P.s_ev_act[dst] = __ldg(P.act + o0 + src);
                long long out_ts;
                if (P.needs_ts) out_ts = (long long)sec[j] * 1000 + t0ms;   // SaseEvent.getEventBoth (SaseEvent.java:94-106)
                else {
                    const long long raw = __ldg(reinterpret_cast<const long long*>(P.ts_ms) + o0 + src);
                    out_ts = evt_pos ? raw : (long long)rel_seconds(raw - t0ms) * 1000 + t0ms;
                }
                P.s_ev_ts[dst] = out_ts;
            }
            if (return_all && i == 0) P.s_occ_nev[Q.occ_base + occ_at + o] = np;
        }
    }
}

// Final placement.  The dense per-candidate counts (d_nocc, d_nev) are scanned in three levels
// (per-block sums -> chunks of 1024 block sums -> chunk sums, + the in-block scan inside the gather), and the
// gather copies each matching trace's staged occurrences to its final, trace-ordered position.
constexpr int GT = 256;

struct GatherParams {
    const int64_t* cand;
    int64_t n;
    const uint32_t* d_cnt;
    const int64_t* d_stage;
    const int64_t* d_stage_occ;  // nullptr without returnAll: the occurrence is staged at the candidate's index
    unsigned long long* blk;  // [3][n_blk] block sums -> exclusive bases inside their chunk of 1024 blocks
    int64_t n_blk;
    unsigned long long* top;  // [3][n_chunks] chunk sums -> exclusive bases
    int64_t n_chunks;
    const int32_t* s_occ_nev;
    const int32_t* s_ev_pos;
    const int32_t* s_ev_rank;
    const int32_t* s_ev_act;
    const int64_t* s_ev_ts;
    RebaseOffsets base;  // added to trace_idx / occ_off / ev_off (chunked evaluation: the chunk's place in the whole result)
    int64_t* trace_idx;
    int64_t* occ_off;
    int64_t* ev_off;
    int32_t* ev_posv;
    int32_t* ev_rank;
    int32_t* ev_act;
    int64_t* ev_ts;
    int all_cols;
    // uniform placement: K1-P's tile words ([2][n_tiles], DetectParams::tile_words) and its fixed staging slots
    const uint32_t* tile_words;
    int64_t n_tiles;
    int64_t fix_ev;
};

template <int NTHR = GT>
__device__ __forceinline__ void block_scan3(unsigned long long v[3], unsigned long long excl[3], unsigned long long tot[3]) {
    __shared__ unsigned long long ws[3][NTHR / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long inc[3] = {v[0], v[1], v[2]};
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            unsigned long long y = __shfl_up_sync(0xffffffffu, inc[q], d);
            if (lane >= d) inc[q] += y;
        }
    if (lane == 31)
        for (int q = 0; q < 3; ++q) ws[q][warp] = inc[q];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        unsigned long long before = 0, all = 0;
        for (int k = 0; k < NTHR / 32; ++k) {
            if (k < warp) before += ws[q][k];
            all += ws[q][k];
        }
        excl[q] = before + inc[q] - v[q];
        tot[q] = all;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(GT) count_blocks_kernel(const __grid_constant__ GatherParams G) {
    const int64_t i = (int64_t)blockIdx.x * GT + threadIdx.x;
    unsigned long long v[3] = {0, 0, 0}, ex[3], tot[3];
    if (i < G.n) {
        const uint32_t w = G.d_cnt[i], c = w & 0xFFFFu;
        v[0] = c ? 1 : 0;
        v[1] = c;
        v[2] = w >> 16;
    }
    block_scan3(v, ex, tot);
    if (threadIdx.x == 0)
        for (int q = 0; q < 3; ++q) G.blk[q * G.n_blk + blockIdx.x] = tot[q];
}

// Exclusive scan of the three rows of block sums in two levels, all loads coalesced: every block of scan_chunks_kernel
// scans one chunk of 1024 sums in place and reports the chunk totals; scan_top_kernel (one block) scans the chunk
// totals; the gather adds blk[block] + top[block / 1024].
constexpr int SC = 1024;
__global__ void __launch_bounds__(SC) scan_chunks_kernel(unsigned long long* blk, int64_t n_blk, unsigned long long* top, int64_t n_chunks) {
    const int64_t i = (int64_t)blockIdx.x * SC + threadIdx.x;
    unsigned long long v[3] = {0, 0, 0}, ex[3], tot[3];
    if (i < n_blk)
#pragma unroll
        for (int q = 0; q < 3; ++q) v[q] = blk[q * n_blk + i];
    block_scan3<SC>(v, ex, tot);
    if (i < n_blk)
#pragma unroll
        for (int q = 0; q < 3; ++q) blk[q * n_blk + i] = ex[q];
    if (threadIdx.x == 0)
#pragma unroll
        for (int q = 0; q < 3; ++q) top[q * n_chunks + blockIdx.x] = tot[q];
}
__global__ void __launch_bounds__(SC) scan_top_kernel(unsigned long long* top, int64_t n_chunks) {
    unsigned long long carry[3] = {0, 0, 0};
    for (int64_t base = 0; base < n_chunks; base += SC) {
        const int64_t i = base + threadIdx.x;
        unsigned long long v[3] = {0, 0, 0}, ex[3], tot[3];
        if (i < n_chunks)
#pragma unroll
            for (int q = 0; q < 3; ++q) v[q] = top[q * n_chunks + i];
        block_scan3<SC>(v, ex, tot);
        if (i < n_chunks)
#pragma unroll
            for (int q = 0; q < 3; ++q) top[q * n_chunks + i] = carry[q] + ex[q];
#pragma unroll
        for (int q = 0; q < 3; ++q) carry[q] += tot[q];
    }
}

__global__ void __launch_bounds__(GT) gather_kernel(const __grid_constant__ GatherParams G) {
    const int64_t i = (int64_t)blockIdx.x * GT + threadIdx.x;
    const int lane = threadIdx.x & 31;
    unsigned long long v[3] = {0, 0, 0}, ex[3], tot[3];
    uint32_t nocc = 0;
    long long se = 0;
    int64_t cand_i = i;
    // everything the placement needs is requested up front (one memory latency instead of four in a row): the block's
    // bases, the staging place (read speculatively: unwritten and unused for a trace without a match), the trace id
    const int64_t chunk = blockIdx.x / SC;
    unsigned long long bb[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) bb[q] = G.top[q * G.n_chunks + chunk] + G.blk[q * G.n_blk + blockIdx.x];
    if (i < G.n) {
        const uint32_t w = G.d_cnt[i];
        se = G.d_stage[i];
        if (G.cand) cand_i = G.cand[i];
        nocc = w & 0xFFFFu;
        v[0] = nocc ? 1 : 0;
        v[1] = nocc;
        v[2] = w >> 16;
    }
    block_scan3(v, ex, tot);
    const int64_t tp = (int64_t)(bb[0] + ex[0]);
    const int64_t op = (int64_t)(bb[1] + ex[1]);
    const int64_t ep = (int64_t)(bb[2] + ex[2]);
    if (nocc) {
        G.trace_idx[tp] = cand_i + G.base.trace;
        G.occ_off[tp] = op + G.base.occ;
        if (G.d_stage_occ) {
            const int64_t so = G.d_stage_occ[i];
            int64_t e = ep;
            for (uint32_t o = 0; o < nocc; ++o) {
                G.ev_off[op + o] = e + G.base.ev;
                e += G.s_occ_nev[so + o];
            }
        } else {
            G.ev_off[op] = ep + G.base.ev;  // one occurrence per trace
        }
    }
    // The events of a warp's 32 candidates are contiguous in the output (ep ascends with the lane) and, per candidate,
    // contiguous in the staging area: copy them as one flat stream, 32 events per step, all four columns coalesced.
    const unsigned my_ev = (unsigned)v[2];
    unsigned incl = my_ev;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
    }
    const unsigned wtot = __shfl_sync(0xffffffffu, incl, 31);
    const long long wbase = shfl_i64(ep, 0);  // lane 0's exclusive base = first output slot of the warp
    for (unsigned f0 = 0; f0 < wtot; f0 += 32) {
        const unsigned f = f0 + lane;
        int lo = 0, hi = 31;
#pragma unroll
        for (int it = 0; it < 5; ++it) {
            const int mid = (lo + hi) >> 1;
            const unsigned vmid = __shfl_sync(0xffffffffu, incl, mid);
            if (vmid > f) hi = mid; else lo = mid + 1;
        }
        const int owner = lo & 31;
        const unsigned o_incl = __shfl_sync(0xffffffffu, incl, owner);
        const unsigned o_ev = __shfl_sync(0xffffffffu, my_ev, owner);
        const long long o_se = shfl_i64(se, owner);
        if (f < wtot) {
            const long long from = o_se + (long long)(f - (o_incl - o_ev));
            const long long to = wbase + f;
            // all loads first: one memory latency per step, not four
            const int32_t c_pos = __ldg(G.s_ev_pos + from);
            int32_t c_rank = 0, c_act = 0;
            long long c_ts = 0;
            if (G.all_cols) {
                c_rank = __ldg(G.s_ev_rank + from);
                c_act = __ldg(G.s_ev_act + from);
                c_ts = __ldg(reinterpret_cast<const long long*>(G.s_ev_ts) + from);
            }
            G.ev_posv[to] = c_pos;
            if (G.all_cols) {
                G.ev_rank[to] = c_rank;
                G.ev_act[to] = c_act;
                G.ev_ts[to] = c_ts;
            }
        }
    }
}

// The compact block of the multi-GPU exchange (layout: pack_layout below).
struct PackSections {
    uint32_t* trace;
    int64_t* base;
    uint32_t *occ_off, *ev_off;
    uint16_t* pos;
    uint8_t* rank;
    uint16_t* act;
    int32_t* delta;
    int64_t* err;
    int64_t* unsup;
    int32_t seconds;
    int* status;
};

// The placement when every matching trace holds ONE occurrence of k events (class NK asked for the first-largest
// occurrence: the metric's configuration), into the result columns (PACK = false) or into the exchange's compact block
// (PACK = true).  One warp per block of 256 candidates, the granularity of the block sums, so its first row is known
// from the scanned sums alone.
//   rows     K1-P left two words per tile of 32 candidates (DetectParams::tile_words): the lanes that matched and the
//            lanes it sent to the overflow list.  Only the overflow lanes read d_cnt / d_stage, which the staged
//            kernels and K1-L wrote for exactly those candidates; a lane's row is the popcount of the matching lanes
//            below it.  Without K1-P every lane is marked overflow, so every candidate is read as the staged kernel left it.
//   events   a K1-P match's k events sit at its tile's fixed slots in lane order, one word {pos, rank, act} and the
//            timestamp each; a re-run trace's at d_stage in the four staged columns.  Where every row of a block comes
//            from K1-P the block's events are 8 contiguous runs; they are copied 128 per step, all loads of a step
//            issued before its first store.
template <bool PACK>
__global__ void __launch_bounds__(GT) gather_uniform_kernel(const __grid_constant__ GatherParams G, const __grid_constant__ PackSections O,
                                                            const int k) {
    __shared__ long long s_src[GT / 32][256];   // per row of the block: K1-P slot (>= 0) or ~d_stage of a re-run trace
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t blk = (int64_t)blockIdx.x * (GT / 32) + warp;
    if (blk >= G.n_blk) return;
    long long* src = s_src[warp];
    const uint32_t below = (1u << lane) - 1u;
    const int64_t t0 = blk * 8;
    // the tile words: lanes 0-7 the matched lanes of the block's tiles, lanes 8-15 the overflow lanes
    uint32_t w = 0;
    if (lane < 16 && t0 + (lane & 7) < G.n_tiles) w = __ldg(G.tile_words + (lane < 8 ? 0 : G.n_tiles) + t0 + (lane & 7));
    const unsigned long long b0 = G.top[blk / SC] + G.blk[blk];   // matching traces before this block (sum 0 of 3)
    uint32_t mw[8], full[8];
    long long se[8];
    uint32_t any_ovf = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        mw[j] = __shfl_sync(0xffffffffu, w, j);
        full[j] = __shfl_sync(0xffffffffu, w, 8 + j);   // (overflow lanes for now)
        any_ovf |= full[j];
        se[j] = 0;
    }
    if (any_ovf) {   // re-run traces in the block (uniform branch)
        uint32_t cnt[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int64_t c = blk * 256 + j * 32 + lane;
            cnt[j] = 0;
            if (((full[j] >> lane) & 1u) && c < G.n) {
                cnt[j] = G.d_cnt[c];
                se[j] = G.d_stage[c];
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) full[j] = mw[j] | __ballot_sync(0xffffffffu, (cnt[j] & 0xFFFFu) != 0);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) full[j] = mw[j];
    }
    // rows: the trace columns, and where each row's events are staged
    unsigned n_rows = 0;
    int bad = 0;
    int64_t cid[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int64_t c = blk * 256 + j * 32 + lane;
        cid[j] = (!PACK && G.cand && ((full[j] >> lane) & 1u)) ? __ldg(G.cand + c) : c;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        if ((full[j] >> lane) & 1u) {
            const unsigned r = n_rows + __popc(full[j] & below);
            src[r] = ((mw[j] >> lane) & 1u) ? G.fix_ev + (t0 + j) * 32 * k + (long long)__popc(mw[j] & below) * k : ~se[j];
            const int64_t tp = (int64_t)b0 + r;
            if constexpr (PACK) {
                bad |= (unsigned long long)cid[j] > 0xFFFFFFFFull;
                O.trace[tp] = (uint32_t)cid[j];   // no candidate list on the exchange path: the shard-local trace index
            } else {
                G.trace_idx[tp] = cid[j] + G.base.trace;
                G.occ_off[tp] = tp + G.base.occ;
                G.ev_off[tp] = tp * k + G.base.ev;
            }
        }
        n_rows += __popc(full[j]);
    }
    __syncwarp();
    const unsigned tot = n_rows * (unsigned)k;   // <= 2048
    const long long ebase = (long long)b0 * k;
    const unsigned inv = 65536u / (unsigned)k + 1u;   // (f * inv) >> 16 == f / k for every f < 2048 and k <= 8
    const long long* s_ts = reinterpret_cast<const long long*>(G.s_ev_ts);
    for (unsigned f0 = 0; f0 < tot; f0 += 128) {
        int32_t v_pos[4], v_rank[4], v_act[4];
        long long v_ts[4], v_t0[4];
        bool packed[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const unsigned f = f0 + 32 * u + lane;
            v_pos[u] = v_rank[u] = v_act[u] = 0;
            v_ts[u] = v_t0[u] = 0;
            packed[u] = true;
            if (f < tot) {
                const unsigned r = (f * inv) >> 16, e = f - r * (unsigned)k;
                long long s = src[r];
                packed[u] = s >= 0;
                if (!packed[u]) s = ~s;
                v_pos[u] = __ldg(G.s_ev_pos + s + e);
                if (G.all_cols) {
                    if (!packed[u]) {
                        v_rank[u] = __ldg(G.s_ev_rank + s + e);
                        v_act[u] = __ldg(G.s_ev_act + s + e);
                    }
                    v_ts[u] = __ldg(s_ts + s + e);
                    if (PACK) v_t0[u] = __ldg(s_ts + s);   // the row's first event: base of the deltas
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const unsigned f = f0 + 32 * u + lane;
            if (f >= tot) continue;
            if (packed[u]) {
                const uint32_t x = (uint32_t)v_pos[u];
                v_pos[u] = (int32_t)(x & 0xFFu);
                v_rank[u] = (int32_t)((x >> 8) & 0xFFu);
                v_act[u] = (int32_t)(x >> 16);
            }
            const long long to = ebase + f;
            if constexpr (PACK) {
                bad |= (unsigned)v_pos[u] > 0xFFFFu;
                O.pos[to] = (uint16_t)v_pos[u];
                if (G.all_cols) {
                    const unsigned r = (f * inv) >> 16;
                    if (f == r * (unsigned)k) O.base[(int64_t)b0 + r] = v_ts[u];
                    long long d = v_ts[u] - v_t0[u];
                    if (O.seconds) {
                        bad |= d % 1000 != 0;
                        d /= 1000;
                    }
                    bad |= (unsigned)v_rank[u] > 0xFFu || (unsigned)v_act[u] > 0xFFFFu || d < -0x7fffffffll - 1 || d > 0x7fffffffll;
                    O.rank[to] = (uint8_t)v_rank[u];
                    O.act[to] = (uint16_t)v_act[u];
                    O.delta[to] = (int32_t)d;
                }
            } else {
                G.ev_posv[to] = v_pos[u];
                if (G.all_cols) {
                    G.ev_rank[to] = v_rank[u];
                    G.ev_act[to] = v_act[u];
                    G.ev_ts[to] = v_ts[u];
                }
            }
        }
    }
    if (PACK && __any_sync(0xffffffffu, bad) && lane == 0) atomicOr(O.status, XST_RANGE);
}

__global__ void set_tail_kernel(int64_t* occ_off, int64_t n_tr, int64_t n_occ, int64_t* ev_off, int64_t n_ev, RebaseOffsets base) {
    occ_off[n_tr] = n_occ + base.occ;
    ev_off[n_occ] = n_ev + base.ev;
}

// ---------------------------------------------------------------------------------- host side
namespace {

// A block of the context's device arena (common.cuh): scratch and results of a request, returned when the request is done.
struct DevBuf {
    void* p = nullptr;
    Ctx* c = nullptr;
    explicit DevBuf(Ctx* ctx) : c(ctx) {}
    DevBuf(const DevBuf&) = delete;
    ~DevBuf() { if (p) dev_arena_free(c, p); }
    int alloc(size_t bytes) {
        if (p) { dev_arena_free(c, p); p = nullptr; }
        p = dev_arena_alloc(c, bytes);
        return p ? SIESTA_OK : SIESTA_E_NOMEM;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
    void* release() { void* q = p; p = nullptr; return q; }
};

// a slice of a DevBuf
struct View {
    void* p;
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

template <int W, int R, int NF, bool SMEM_RUNS, int MODE>
int launch_detect(const Ctx* ctx, cudaStream_t stream, DetectParams P, const DevNfa& nfa) {
    typedef WarpSmem<W, R, NF, SMEM_RUNS> L;
    const bool needs_aux = MODE == FAST_NK && (P.flags & SIESTA_F_RETURN_ALL) != 0;
    int nt = NT;
    if (const char* env = std::getenv("SIESTA_K1_THREADS")) {  // tuning aid: threads per CTA (multiple of 32, <= NT)
        const int v = std::atoi(env);
        if (v >= 32 && v <= NT_MAX && v % 32 == 0) nt = v;
    }
    const size_t smem = L::total(needs_aux) * (nt / 32);
    auto kern = detect_kernel<W, R, NF, SMEM_RUNS, MODE>;
    SIESTA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (const char* env = std::getenv("SIESTA_K1_CARVEOUT")) {  // tuning aid: shared-memory carveout in percent
        const int v = std::atoi(env);
        if (v >= 0 && v <= 100) SIESTA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    }
    int per_sm = 0;
    SIESTA_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt, smem));
    if (per_sm < 1) per_sm = 1;
    const int64_t n_tiles = (P.n_work + 31) / 32;   // one tile = the 32 traces of one warp (upper bound if the count is on the device)
    const int64_t ctas_needed = (n_tiles + nt / 32 - 1) / (nt / 32);
    if (const char* env = std::getenv("SIESTA_K1_CTAS_PER_SM")) {  // tuning aid: cap on resident CTAs per SM
        const int v = std::atoi(env);
        if (v >= 1 && v < per_sm) per_sm = v;
    }
    int grid = (int)std::min<int64_t>(ctas_needed, (int64_t)ctx->sm_count * per_sm);
    // a re-run launch (work count on the device: the traces the previous kernel could not hold) usually finds nothing to do;
    // two CTAs per SM start and end in a few microseconds and still take any list through the tile counter
    if (P.n_work_dev) grid = std::min(grid, ctx->sm_count * 2);
    if (grid < 1) grid = 1;
    kern<<<grid, nt, smem, stream>>>(P, nfa);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

}  // namespace

// A verification request between its two halves (siesta_detect_device_begin / _finish): everything the second half
// needs.  The first half enqueues the verification kernels and the copy of the counters and returns without waiting;
// the second half waits for the counters, allocates the result and enqueues the placement.  A caller with several
// requests in flight (a server, the multi-GPU bench) issues the next request's first half before it exchanges the
// results of the previous one, so the host-side work of one request overlaps the scan of the next.
struct DetectPending {
    Log* log = nullptr;
    cudaStream_t stream = nullptr;
    int64_t n = 0;
    uint32_t flags = 0;
    RebaseOffsets base{0, 0, 0};
    const int64_t* d_cand = nullptr;
    DetectParams P;
    size_t n_blk = 0;
    unsigned long long *d_blk = nullptr, *d_top = nullptr, *d_counters = nullptr;
    int64_t* d_err = nullptr;
    int64_t* d_unsup = nullptr;           // candidate indices of the traces beyond the engine limits
    int unsup_slot = 7;                   // counter that counts them (7: wide launch, 14: K1-L)
    void* work = nullptr;                 // scratch of the call (freed by the second half)
    int uniform_k = 0;                    // > 0: one occurrence per trace, uniform_k events each (class NK, first-largest)
    const uint32_t* tile_words = nullptr; // set: the uniform placement (gather_uniform_kernel) places the result
    int64_t n_tiles = 0, fix_ev = 0;
    cudaEvent_t ev0 = nullptr, evd = nullptr;
    unsigned long long* h_cnt = nullptr;  // pinned, 16 words
    const uint16_t* d_lut = nullptr;      // the request's tables on the device (a later block of the same request reuses them)
    const uint4* d_nkp_lut = nullptr;
};

static unsigned long long* pinned_counters_get(Ctx* c) {
    std::lock_guard<std::mutex> g(c->arena_mu);
    if (c->pinned_counters.empty()) {
        void* slab = nullptr;
        if (cudaHostAlloc(&slab, 32 * 128, cudaHostAllocDefault) != cudaSuccess) return nullptr;
        c->pinned_slabs.push_back(slab);
        for (int i = 0; i < 32; ++i) c->pinned_counters.push_back(reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(slab) + 128 * i));
    }
    unsigned long long* p = c->pinned_counters.back();
    c->pinned_counters.pop_back();
    return p;
}
static void pinned_counters_put(Ctx* c, unsigned long long* p) {
    if (!p) return;
    std::lock_guard<std::mutex> g(c->arena_mu);
    c->pinned_counters.push_back(p);
}

static void pending_discard(DetectPending* q) {
    if (!q) return;
    if (q->work) dev_arena_free(q->log->ctx, q->work);   // (every caller has waited for the request's stream)
    if (q->ev0) cudaEventDestroy(q->ev0);
    if (q->evd) cudaEventDestroy(q->evd);
    pinned_counters_put(q->log->ctx, q->h_cnt);
    delete q;
}

int detect_device_finish_impl(DetectPending* q, siesta_dev_matches* out);

int detect_device_begin_impl(Log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand, uint32_t flags,
                             cudaStream_t stream, RebaseOffsets base, DetectPending** pending, const DetectPending* sibling) {
    // sibling: an earlier block of the SAME request (same NFA, flags, alphabet) on the exchange path - its device tables
    // are reused and the counters are not copied to the host (the placement reads them on the device), so the block adds
    // no copy to the stream and the host runs ahead of the device.
    *pending = nullptr;
    base.trace += log->first_trace;
    DevNfa dn;
    int rc = validate_nfa(nfa, flags, &dn);
    if (rc != SIESTA_OK) return rc;
    const Ctx* ctx = log->ctx;
    SIESTA_CUDA_OK(cudaSetDevice(ctx->device));
    if (!stream) stream = ctx->stream;
    const int64_t n = d_cand ? n_cand : log->n_traces;
    const bool return_all = (flags & SIESTA_F_RETURN_ALL) != 0;
    const bool all_cols = (flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;

    std::vector<uint16_t> lut;
    int needs_ts = 0, n_positive = 0;
    build_lut(nfa, dn, log->n_activities, flags, lut, &needs_ts, &n_positive);

    // staging bounds: selected occurrences of a trace are disjoint, so their events never exceed the
    // trace's filtered events (<= 64 on the widest engine configuration)
    const int64_t wide = std::min<int64_t>(log->n_events, n * 64);
    const int64_t cap_occ = return_all ? wide : n;
    const int uniform_k = (!return_all && !dn.any_kleene) ? std::max(1, n_positive) : 0;
    const int64_t cap_ev = uniform_k ? n * uniform_k : wide;

    // one stream-ordered allocation for all scratch of the call, carved by a bump pointer
    DevBuf work(log->ctx);
    const size_t nn = (size_t)std::max<int64_t>(n, 1);
    size_t w_off = 0;
    auto carve = [&w_off](size_t bytes) {
        const size_t at = w_off;
        w_off += (bytes + 255) & ~(size_t)255;
        return at;
    };
    // class NK, first-largest only, no relative seconds: the raw-slot kernel K1-P goes first (its overflow list feeds
    // the staged kernel).  Decided before the scratch is carved: it needs a second overflow list.
    // K1-P numbers CLASSES by state-membership signature (activities of one `or` state share a class), so more patterns
    // fit three planes than with one class per activity; it re-reads the activity id of the few reported events.
    NkwProgram prog;
    const int nkw_space = nkw_build(dn, flags, &prog);
    std::vector<uint16_t> sigs;   // distinct signatures, class c = sigs[c - 1]
    for (size_t a = 0; a < lut.size(); ++a) {
        const uint16_t sg = lut[a] & 0xFFu;
        if (sg && std::find(sigs.begin(), sigs.end(), sg) == sigs.end()) sigs.push_back(sg);
    }
    // (nkw_build only admits predicates that read no relative seconds; with returnAll the seconds are needed by the overlap
    //  test alone, and the traces that need it - more than one engine match - are re-run on the staged kernel)
    const bool use_nkp = nkw_space != NKW_NONE && (!needs_ts || return_all) && log->act_valid && log->n_activities <= 255 && !sigs.empty() && sigs.size() <= 7 &&
                         (reinterpret_cast<uintptr_t>(log->d_act) & 31u) == 0 && std::getenv("SIESTA_K1_NO_NKP") == nullptr;   // (keep in step with detect_nkp_eligible)
    // staging regions: [0, cap_ev) by atomics (staged kernels), then K1-P's fixed tile slots (n_positive per candidate: with
    // returnAll cap_ev is bounded by the log's events, which may be fewer), then K1-L's
    const size_t reg2 = use_nkp ? (size_t)std::max<int64_t>(cap_ev, n * (int64_t)std::max(1, n_positive)) : 0;
    // returnAll: K1-P answers the traces with ONE engine match (its occurrence is the selection) and stages that occurrence's
    // event count in a slot of its own per candidate, behind the staged kernels' and K1-L's
    // class NK: the traces beyond the mask kernels' limits re-run on K1-L, which stages in a region of its own behind
    // the others and takes its per-trace arrays from a pool
    const bool use_long = dn.fast_class == FAST_NK && std::getenv("SIESTA_K1_NO_LONG") == nullptr;
    const int64_t cap_long = use_long ? std::min<int64_t>(log->n_events, (int64_t)1 << 21) : 0;
    const size_t long_pool = use_long ? (size_t)std::min<int64_t>(std::max<int64_t>(log->n_events * 64, (int64_t)1 << 20), (int64_t)256 << 20) : 0;
    const size_t n_blk = (nn + GT - 1) / GT;
    // a uniform result is placed by gather_uniform_kernel from two words per tile of 32 candidates
    const bool uniform_place = uniform_k > 0 && uniform_k <= 8 && std::getenv("SIESTA_NO_UNIFORM_GATHER") == nullptr;
    const size_t n_tiles = (nn + 31) / 32;
    const size_t o_tiles = uniform_place ? carve(n_tiles * 2 * 4) : 0;
    const size_t o_ovf2 = use_nkp ? carve(nn * 8) : 0;
    const size_t o_unsup = carve((size_t)SIESTA_MAX_UNSUPPORTED * 8);   // traces beyond the engine limits (wide launch)
    const size_t o_unsup2 = use_long ? carve((size_t)SIESTA_MAX_UNSUPPORTED * 8) : 0;   // ... and beyond K1-L's pool / staging
    const size_t o_pool = carve(long_pool);
    const size_t o_nlut = use_nkp ? carve((size_t)(log->n_activities + 1) * 16) : 0;
    const size_t o_lut = carve(lut.size() * sizeof(uint16_t)), o_nocc = carve(nn * 4), o_stage = carve(nn * 8),
                 o_stage_occ = carve(return_all ? nn * 8 : 0), o_counters = carve(32 * 8), o_err = carve(nn * 8), o_ovf = carve(nn * 8),
                 o_blk = carve(n_blk * 3 * 8), o_top = carve(((n_blk + 1023) / 1024) * 3 * 8), o_occ_nev = carve(return_all ? ((size_t)(cap_occ + cap_long) + (use_nkp ? nn : 0)) * 4 : 0), o_pos = carve(((size_t)cap_ev + reg2 + (size_t)cap_long) * 4);
    size_t o_rank = 0, o_act = 0, o_ts = 0;
    if (all_cols) {
        o_rank = carve(((size_t)cap_ev + reg2 + (size_t)cap_long) * 4);
        o_act = carve(((size_t)cap_ev + reg2 + (size_t)cap_long) * 4);
        o_ts = carve(((size_t)cap_ev + reg2 + (size_t)cap_long) * 8);
    }
    if ((rc = work.alloc(w_off))) return rc;
    char* wb = work.as<char>();
    const View b_lut{wb + o_lut}, b_nocc{wb + o_nocc}, b_stage{wb + o_stage}, b_stage_occ{wb + o_stage_occ},
        b_counters{wb + o_counters}, b_err{wb + o_err}, b_ovf{wb + o_ovf}, b_blk{wb + o_blk}, s_occ_nev{wb + o_occ_nev},
        s_ev_pos{wb + o_pos}, s_ev_rank{all_cols ? wb + o_rank : nullptr}, s_ev_act{all_cols ? wb + o_act : nullptr},
        s_ev_ts{all_cols ? wb + o_ts : nullptr};

    cudaEvent_t ev0 = nullptr, evd = nullptr;
    SIESTA_CUDA_OK(cudaEventCreate(&ev0));
    SIESTA_CUDA_OK(cudaEventCreate(&evd));
    unsigned long long* h_cnt = nullptr;
    const uint4* d_nkp_lut = nullptr;
    struct BeginGuard {   // an error return of the first half releases what it holds so far
        cudaEvent_t &a, &b;
        unsigned long long*& h;
        Ctx* c;
        bool armed;
        ~BeginGuard() {
            if (!armed) return;
            if (a) cudaEventDestroy(a);
            if (b) cudaEventDestroy(b);
            pinned_counters_put(c, h);
        }
    } begin_guard{ev0, evd, h_cnt, log->ctx, true};
    if (!sibling) SIESTA_CUDA_OK(cudaMemcpyAsync(b_lut.p, lut.data(), lut.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, stream));
    SIESTA_CUDA_OK(cudaMemsetAsync(b_counters.p, 0, 256, stream));
    SIESTA_CUDA_OK(cudaMemsetAsync(b_blk.p, 0, n_blk * 3 * 8, stream));
    SIESTA_CUDA_OK(cudaEventRecord(ev0, stream));

    DetectParams P;
    std::memset(&P, 0, sizeof(P));
    P.trace_off = log->d_trace_off;
    P.act = log->d_act;
    P.ts_ms = log->d_ts_ms;
    P.cand = d_cand;
    P.work = nullptr;
    P.n_work = n;
    P.lut = sibling ? sibling->d_lut : b_lut.as<uint16_t>();
    P.n_act = log->n_activities;
    P.n_events = log->n_events;
    // classes: the pattern's activities numbered 1..K
    P.alpha_mode = !log->act_valid ? 2 : (log->n_activities <= 32 ? 0 : (log->n_activities <= 64 ? 1 : 2));
    std::memset(P.relrev, 0, sizeof(P.relrev));
    std::memset(P.cls_word, 0, sizeof(P.cls_word));
    std::memset(P.cls_act, 0, sizeof(P.cls_act));
    P.n_planes = 1;
    if (P.alpha_mode != 2) {
        int K = 0;
        for (size_t a = 0; a < lut.size(); ++a) K += lut[a] != 0;
        if (K > 7) P.alpha_mode = 2;
        else {
            int c = 0;
            for (size_t a = 0; a < lut.size(); ++a) {
                if (!lut[a]) continue;
                ++c;
                P.cls_word[c] = lut[a];
                P.cls_act[c] = (int32_t)a;
                for (int p = 0; p < 3; ++p)
                    if ((c >> p) & 1) P.relrev[p][a >> 5] |= 0x80000000u >> (a & 31);
            }
            P.n_planes = K <= 1 ? 1 : (K <= 3 ? 2 : 3);
        }
    }
    P.vec_ok = (reinterpret_cast<uintptr_t>(log->d_act) & 15u) == 0 ? 1 : 0;
    P.flags = flags;
    P.needs_ts = needs_ts;
    P.d_cnt = b_nocc.as<uint32_t>();
    P.d_stage = b_stage.as<int64_t>();
    P.d_stage_occ = b_stage_occ.as<int64_t>();
    P.s_occ_nev = s_occ_nev.as<int32_t>();
    P.s_ev_pos = s_ev_pos.as<int32_t>();
    P.s_ev_rank = s_ev_rank.as<int32_t>();
    P.s_ev_act = s_ev_act.as<int32_t>();
    P.s_ev_ts = s_ev_ts.as<int64_t>();
    P.cap_occ = cap_occ;
    P.cap_ev = cap_ev;
    P.counters = b_counters.as<unsigned long long>();
    P.err_list = b_err.as<int64_t>();
    P.ovf_list = b_ovf.as<int64_t>();
    P.blk_sums = b_blk.as<unsigned long long>();
    P.n_blk = (int64_t)n_blk;

    P.ovf_slot = 4;
    P.tile_slot = 16;   // the tile counters live on their own 128-byte line (slots 16..)
    h_cnt = pinned_counters_get(log->ctx);
    if (!h_cnt) {
        set_error("cudaHostAlloc (counters) failed");
        return SIESTA_E_NOMEM;
    }
    std::memset(h_cnt, 0, 128);
    uint32_t* tile_words = uniform_place ? reinterpret_cast<uint32_t*>(wb + o_tiles) : nullptr;
    if (n > 0) {
        if (uniform_place && !use_nkp) {   // no K1-P: every lane is an overflow lane, its d_cnt is read
            SIESTA_CUDA_OK(cudaMemsetAsync(tile_words, 0, n_tiles * 4, stream));
            SIESTA_CUDA_OK(cudaMemsetAsync(tile_words + n_tiles, 0xFF, n_tiles * 4, stream));
        }
        if (use_nkp) {
            DetectParams N = P;
            N.tile_words = tile_words;
            N.ovf_list = reinterpret_cast<int64_t*>(wb + o_ovf2);
            N.ovf_slot = 13;
            N.tile_slot = 18;
            N.fix_ev = cap_ev;
            N.fix_np = std::max(1, n_positive);
            N.fix_occ = return_all ? cap_occ + cap_long : -1;
            // the scan's table: {m, b0, b1, b2} per activity (detect_nkp.cu); class c = index of the signature + 1
            std::vector<uint32_t> nlut((size_t)(log->n_activities + 1) * 4, 0u);
            std::memset(N.cls_word, 0, sizeof(N.cls_word));
            for (int a = 0; a <= log->n_activities; ++a) {
                const uint16_t sg = a < log->n_activities ? (lut[a] & 0xFFu) : 0;
                int c = 0;
                if (sg) {
                    c = (int)(std::find(sigs.begin(), sigs.end(), sg) - sigs.begin()) + 1;
                    N.cls_word[c] = sg;
                }
                nlut[4 * a + 0] = (nkw_space == NKW_RAW || c) ? 2u : 1u;
                for (int p = 0; p < 3; ++p) nlut[4 * a + 1 + p] = (c >> p) & 1;
            }
            if (sibling && sibling->d_nkp_lut) N.nkp_lut = sibling->d_nkp_lut;
            else {
                SIESTA_CUDA_OK(cudaMemcpyAsync(wb + o_nlut, nlut.data(), nlut.size() * 4, cudaMemcpyHostToDevice, stream));
                N.nkp_lut = reinterpret_cast<const uint4*>(wb + o_nlut);
            }
            d_nkp_lut = N.nkp_lut;
            N.n_planes = sigs.size() <= 1 ? 1 : (sigs.size() <= 3 ? 2 : 3);
            std::memset(N.st_inv, 0, sizeof(N.st_inv));
            std::memset(N.st_single, 0, sizeof(N.st_single));
            for (int k = 0; k < nfa->n_states; ++k) {
                int n_own = 0, c_own = 0;
                for (int c = 1; c <= (int)sigs.size(); ++c)
                    if (sigs[(size_t)c - 1] & (1u << k)) {
                        ++n_own;
                        c_own = c;
                    }
                if (n_own == 1) {
                    N.st_single[k] = 1;
                    for (int p = 0; p < 3; ++p) N.st_inv[k][p] = ((c_own >> p) & 1) ? 0u : 0xFFFFFFFFu;
                }
            }
            if ((rc = launch_nkp(ctx, stream, N, prog, nkw_space))) return rc;
            // the staged kernel below re-runs the traces that did not fit 64 slots (count read from the device)
            P.work = N.ovf_list;
            P.n_work_dev = b_counters.as<unsigned long long>() + 13;
        }
        if (dn.fast_class == FAST_FK2) rc = launch_detect<1, 0, 0, false, FAST_FK2>(ctx, stream, P, dn);
        else if (dn.fast_class == FAST_NK) rc = launch_detect<1, 0, 0, false, FAST_NK>(ctx, stream, P, dn);
        else if (dn.fast_class == FAST_NP1) rc = launch_detect<1, 0, 0, false, FAST_NP1>(ctx, stream, P, dn);
        else rc = launch_detect<1, 16, 16, true, FAST_NONE>(ctx, stream, P, dn);
        if (rc) return rc;
        SIESTA_CUDA_OK(cudaEventRecord(evd, stream));
        // Traces beyond the narrow configuration (24 relevant events; run-list engine: 16 live runs / 16 live families)
        // re-run on the wide one.  The launch is unconditional and reads its work count from the device, so the host
        // does not have to wait for the narrow launch first; with nothing to do it costs a few microseconds.
        DetectParams Q = P;
        Q.work = b_ovf.as<int64_t>();
        Q.n_work_dev = b_counters.as<unsigned long long>() + 4;
        Q.ovf_list = reinterpret_cast<int64_t*>(wb + o_unsup);
        Q.ovf_cap = SIESTA_MAX_UNSUPPORTED;
        Q.ovf_slot = 7;
        Q.tile_slot = 17;
        if (dn.fast_class == FAST_FK2) rc = launch_detect<2, 0, 0, false, FAST_FK2>(ctx, stream, Q, dn);
        else if (dn.fast_class == FAST_NK) rc = launch_detect<2, 0, 0, false, FAST_NK>(ctx, stream, Q, dn);
        else if (dn.fast_class == FAST_NP1) rc = launch_detect<2, 0, 0, false, FAST_NP1>(ctx, stream, Q, dn);
        else rc = launch_detect<2, 1024, 128, false, FAST_NONE>(ctx, stream, Q, dn);
        if (rc) return rc;
        if (use_long) {
            LongParams LQ;
            std::memset(&LQ, 0, sizeof(LQ));
            LQ.work = reinterpret_cast<const int64_t*>(wb + o_unsup);
            LQ.n_work_dev = b_counters.as<unsigned long long>() + 7;
            LQ.work_cap = SIESTA_MAX_UNSUPPORTED;
            LQ.pool = wb + o_pool;
            LQ.pool_bytes = long_pool;
            LQ.ev_base = (int64_t)cap_ev + (int64_t)reg2;
            LQ.ev_cap = cap_long;
            LQ.occ_base = cap_occ;
            LQ.occ_cap = cap_long;
            LQ.unsup = reinterpret_cast<int64_t*>(wb + o_unsup2);
            LQ.unsup_cap = SIESTA_MAX_UNSUPPORTED;
            LQ.n_positive = std::max(1, n_positive);
            detect_long_kernel<<<ctx->sm_count * 2, 128, 0, stream>>>(P, LQ, dn);
            SIESTA_LAUNCHED();
            SIESTA_CUDA_OK(cudaGetLastError());
        }
        if (!sibling) SIESTA_CUDA_OK(cudaMemcpyAsync(h_cnt, b_counters.p, 128, cudaMemcpyDeviceToHost, stream));
    }
    // ---- end of the first half: nothing above waits for the device
    DetectPending* q = new DetectPending();
    q->log = log;
    q->stream = stream;
    q->n = n;
    q->flags = flags;
    q->base = base;
    q->d_cand = d_cand;
    q->P = P;
    q->n_blk = n_blk;
    q->d_blk = b_blk.as<unsigned long long>();
    q->d_top = reinterpret_cast<unsigned long long*>(wb + o_top);
    q->d_counters = b_counters.as<unsigned long long>();
    q->d_err = b_err.as<int64_t>();
    q->d_unsup = reinterpret_cast<int64_t*>(wb + (use_long ? o_unsup2 : o_unsup));
    q->unsup_slot = use_long ? 14 : 7;
    q->work = work.release();
    q->uniform_k = uniform_k;
    q->tile_words = tile_words;
    q->n_tiles = (int64_t)n_tiles;
    q->fix_ev = cap_ev;
    q->ev0 = ev0;
    q->evd = evd;
    q->h_cnt = h_cnt;
    q->d_lut = P.lut;
    q->d_nkp_lut = d_nkp_lut;
    begin_guard.armed = false;
    *pending = q;
    return SIESTA_OK;
}

// Second half: waits for the counters of the first half, allocates the result, enqueues the placement and waits for it.
// Consumes (frees) the pending request whatever the outcome.
int detect_device_finish_impl(DetectPending* q, siesta_dev_matches* out) {
    std::memset(out, 0, sizeof(*out));
    struct Guard {
        DetectPending* q;
        ~Guard() { pending_discard(q); }
    } guard{q};
    Log* log = q->log;
    const Ctx* ctx = log->ctx;
    SIESTA_CUDA_OK(cudaSetDevice(ctx->device));
    cudaStream_t stream = q->stream;
    const int64_t n = q->n;
    const uint32_t flags = q->flags;
    const bool return_all = (flags & SIESTA_F_RETURN_ALL) != 0;
    const bool all_cols = (flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;
    const RebaseOffsets base = q->base;
    const int64_t* d_cand = q->d_cand;
    const DetectParams& P = q->P;
    const size_t n_blk = q->n_blk;
    unsigned long long* h_cnt = q->h_cnt;
    cudaEvent_t ev0 = q->ev0, evd = q->evd, ev1;
    int rc = SIESTA_OK;
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    if (n > 0) {
        if (h_cnt[7] > SIESTA_MAX_UNSUPPORTED || h_cnt[q->unsup_slot] > SIESTA_MAX_UNSUPPORTED) {
            set_error(std::to_string(h_cnt[7]) + " traces exceed the engine limits (64 pattern-relevant events, 1024 live runs or "
                      "65536 events per trace); at most " + std::to_string(SIESTA_MAX_UNSUPPORTED) + " are listed per request");
            return SIESTA_E_UNSUPPORTED;
        }
        if (h_cnt[5] > 0) {
            set_error("internal: occurrence staging overflow");
            return SIESTA_E_NOMEM;
        }
    }
    SIESTA_CUDA_OK(cudaEventCreate(&ev1));
    struct EvGuard {
        cudaEvent_t e;
        ~EvGuard() { cudaEventDestroy(e); }
    } ev1_guard{ev1};
#ifdef SIESTA_PHASE_TIMING
    fprintf(stderr, "[siesta phase timing] warp-cycles: filter %llu engine %llu output %llu\n", h_cnt[8], h_cnt[9], h_cnt[10]);
#endif
    const int64_t n_occ = (int64_t)h_cnt[0], n_ev = (int64_t)h_cnt[1], n_tr = (int64_t)h_cnt[6], n_err = (int64_t)h_cnt[3];
    const int64_t n_unsup = n > 0 ? (int64_t)h_cnt[q->unsup_slot] : 0;

    // the result columns: one allocation, owned by the returned object
    DevBuf fin(log->ctx);
    size_t f_off = 0;
    auto fcarve = [&f_off](size_t bytes) {
        const size_t at = f_off;
        f_off += (bytes + 255) & ~(size_t)255;
        return at;
    };
    const size_t q_trace = fcarve((size_t)n_tr * 8), q_occ = fcarve((size_t)(n_tr + 1) * 8), q_evoff = fcarve((size_t)(n_occ + 1) * 8),
                 q_pos = fcarve((size_t)n_ev * 4), q_err = fcarve((size_t)n_err * 8);
    size_t q_rank = 0, q_act = 0, q_ts = 0;
    if (all_cols) {
        q_rank = fcarve((size_t)n_ev * 4);
        q_act = fcarve((size_t)n_ev * 4);
        q_ts = fcarve((size_t)n_ev * 8);
    }
    const size_t q_unsup = fcarve((size_t)n_unsup * 8);
    if ((rc = fin.alloc(f_off))) return rc;
    char* fb = fin.as<char>();
    const View f_unsup{fb + q_unsup};
    const View f_trace{fb + q_trace}, f_occ_off{fb + q_occ}, f_ev_off{fb + q_evoff}, f_pos{fb + q_pos}, f_err{fb + q_err},
        f_rank{all_cols ? fb + q_rank : nullptr}, f_act{all_cols ? fb + q_act : nullptr}, f_ts{all_cols ? fb + q_ts : nullptr};

    if (n > 0) {
        GatherParams G;
        std::memset(&G, 0, sizeof(G));
        G.cand = d_cand;
        G.base = base;
        G.n = n;
        G.d_cnt = P.d_cnt;
        G.d_stage = P.d_stage;
        G.d_stage_occ = return_all ? P.d_stage_occ : nullptr;
        G.n_blk = (int64_t)n_blk;
        G.blk = q->d_blk;
        G.n_chunks = (int64_t)((n_blk + 1023) / 1024);
        G.top = q->d_top;
        G.s_occ_nev = P.s_occ_nev;
        G.s_ev_pos = P.s_ev_pos;
        G.s_ev_rank = P.s_ev_rank;
        G.s_ev_act = P.s_ev_act;
        G.s_ev_ts = P.s_ev_ts;
        G.trace_idx = f_trace.as<int64_t>();
        G.occ_off = f_occ_off.as<int64_t>();
        G.ev_off = f_ev_off.as<int64_t>();
        G.ev_posv = f_pos.as<int32_t>();
        G.ev_rank = f_rank.as<int32_t>();
        G.ev_act = f_act.as<int32_t>();
        G.ev_ts = f_ts.as<int64_t>();
        G.all_cols = all_cols ? 1 : 0;
        G.tile_words = q->tile_words;
        G.n_tiles = q->n_tiles;
        G.fix_ev = q->fix_ev;
        // (the block sums were accumulated by the verification kernels: no counting pass)
        scan_chunks_kernel<<<(unsigned)G.n_chunks, SC, 0, stream>>>(G.blk, G.n_blk, G.top, G.n_chunks);
        SIESTA_LAUNCHED();
        scan_top_kernel<<<1, SC, 0, stream>>>(G.top, G.n_chunks);
        SIESTA_LAUNCHED();
        if (q->tile_words) {
            PackSections none;
            std::memset(&none, 0, sizeof(none));
            gather_uniform_kernel<false><<<(unsigned)((G.n_blk + GT / 32 - 1) / (GT / 32)), GT, 0, stream>>>(G, none, q->uniform_k);
        } else
            gather_kernel<<<(unsigned)G.n_blk, GT, 0, stream>>>(G);
        SIESTA_LAUNCHED();
        SIESTA_CUDA_OK(cudaGetLastError());
    }
    set_tail_kernel<<<1, 1, 0, stream>>>(f_occ_off.as<int64_t>(), n_tr, n_occ, f_ev_off.as<int64_t>(), n_ev, base);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaEventRecord(ev1, stream));
    if (n_err > 0) {  // order the (rare) error list
        std::vector<int64_t> h((size_t)n_err);
        SIESTA_CUDA_OK(cudaMemcpyAsync(h.data(), q->d_err, (size_t)n_err * 8, cudaMemcpyDeviceToHost, stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
        std::sort(h.begin(), h.end());
        for (int64_t& x : h) x += base.trace;
        SIESTA_CUDA_OK(cudaMemcpyAsync(f_err.p, h.data(), (size_t)n_err * 8, cudaMemcpyHostToDevice, stream));
    }
    if (n_unsup > 0) {  // the traces beyond the engine limits, ascending global indices
        std::vector<int64_t> h((size_t)n_unsup);
        SIESTA_CUDA_OK(cudaMemcpyAsync(h.data(), q->d_unsup, (size_t)n_unsup * 8, cudaMemcpyDeviceToHost, stream));
        SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
        if (d_cand) {       // list entries index the candidate list
            std::vector<int64_t> hc((size_t)n_unsup);
            for (int64_t i = 0; i < n_unsup; ++i)
                SIESTA_CUDA_OK(cudaMemcpyAsync(&hc[(size_t)i], d_cand + h[(size_t)i], 8, cudaMemcpyDeviceToHost, stream));
            SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
            h.swap(hc);
        }
        std::sort(h.begin(), h.end());
        for (int64_t& x : h) x += base.trace;
        SIESTA_CUDA_OK(cudaMemcpyAsync(f_unsup.p, h.data(), (size_t)n_unsup * 8, cudaMemcpyHostToDevice, stream));
    }
    SIESTA_CUDA_OK(cudaStreamSynchronize(stream));
    float ms = 0.f, dms = 0.f;
    SIESTA_CUDA_OK(cudaEventElapsedTime(&ms, ev0, ev1));
    if (n > 0) SIESTA_CUDA_OK(cudaEventElapsedTime(&dms, ev0, evd));
    // (the events and the scratch are released by the guards)

    DevMatchesImpl* impl = new DevMatchesImpl();
    out->n_traces = n_tr;
    out->n_occurrences = n_occ;
    out->n_events = n_ev;
    const bool counted = (flags & (SIESTA_F_COUNT_MATCHES | SIESTA_F_RETURN_ALL | SIESTA_F_LITERAL_RUNS)) != 0;
    out->n_matches_emitted = counted ? (int64_t)h_cnt[2] : -1;
    out->n_ref_errors = n_err;
    out->kernel_ms = ms;
    out->detect_ms = dms;
    impl->owner = log->ctx;
    out->d_trace_idx = f_trace.as<int64_t>();
    out->d_occ_off = f_occ_off.as<int64_t>();
    out->d_ev_off = f_ev_off.as<int64_t>();
    out->d_ev_pos = f_pos.as<int32_t>();
    out->d_ev_rank = f_rank.as<int32_t>();
    out->d_ev_act = f_act.as<int32_t>();
    out->d_ev_ts_ms = f_ts.as<int64_t>();
    out->d_err_trace_idx = f_err.as<int64_t>();
    out->n_unsupported = n_unsup;
    out->d_unsupported_trace_idx = f_unsup.as<int64_t>();
    out->block_bytes = (int64_t)f_off;
    impl->block = out->d_block = fin.release();
    out->impl = impl;
    return SIESTA_OK;
}

// ---------------------------------------------------------------------------------- packed placement (multi-GPU exchange)
// The exchange (multi.cu) ships a rank's match list in a compact block.  Here the placement writes that block DIRECTLY
// into the rank's exchange region - no intermediate result, no host wait for the sizes: the sections sit at offsets
// derived from the request's CAPACITY (known before the scan), the actual sizes travel in the block's header.
//   trace    u32[n_tr]  shard-local trace index            base   i64[n_tr]  ev_ts_ms of the trace's first reported event
//   occ_off  u32[n_tr+1], ev_off u32[n_occ+1]              only when uniform_k == 0 (else one occurrence per trace,
//                                                           uniform_k events per occurrence: offsets are arithmetic)
//   pos u16[n_ev]  rank u8[n_ev]  act u16[n_ev]  delta i32[n_ev]  (ev_ts_ms - base) in seconds (EventTs route: exact,
//                                                           both are rel_s * 1000 + t0) or milliseconds (EventPos route)
//   err      i64[n_err] shard-local indices of the traces on which the Java engine would throw (<= XCHG_ERR_CAP)
static inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }
// byte offsets of the sections inside the data area, from the capacities; returns the bytes needed
static size_t pack_layout(int64_t n, int64_t cap_occ, int64_t cap_ev, int uniform_k, bool all_cols, XHeader* h) {
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += al256(bytes); return (int64_t)at; };
    h->o_trace = take((size_t)n * 4);
    h->o_base = all_cols ? take((size_t)n * 8) : 0;
    h->o_occ_off = uniform_k ? 0 : take((size_t)(n + 1) * 4);
    h->o_ev_off = uniform_k ? 0 : take((size_t)(cap_occ + 1) * 4);
    h->o_pos = take((size_t)cap_ev * 2);
    h->o_rank = all_cols ? take((size_t)cap_ev) : 0;
    h->o_act = all_cols ? take((size_t)cap_ev * 2) : 0;
    h->o_delta = all_cols ? take((size_t)cap_ev * 4) : 0;
    h->o_err = take((size_t)XCHG_ERR_CAP * 8);
    h->o_unsup = take((size_t)XCHG_ERR_CAP * 8);
    return o;
}

__global__ void __launch_bounds__(GT) gather_packed_kernel(const __grid_constant__ GatherParams G, const __grid_constant__ PackSections O, int uniform) {
    const int64_t i = (int64_t)blockIdx.x * GT + threadIdx.x;
    const int lane = threadIdx.x & 31;
    unsigned long long v[3] = {0, 0, 0}, ex[3], tot[3];
    uint32_t nocc = 0;
    long long se = 0;
    const int64_t chunk = blockIdx.x / SC;
    unsigned long long bb[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) bb[q] = G.top[q * G.n_chunks + chunk] + G.blk[q * G.n_blk + blockIdx.x];
    if (i < G.n) {
        const uint32_t w = G.d_cnt[i];
        se = G.d_stage[i];
        nocc = w & 0xFFFFu;
        v[0] = nocc ? 1 : 0;
        v[1] = nocc;
        v[2] = w >> 16;
    }
    block_scan3(v, ex, tot);
    const int64_t tp = (int64_t)(bb[0] + ex[0]);
    const int64_t op = (int64_t)(bb[1] + ex[1]);
    const int64_t ep = (int64_t)(bb[2] + ex[2]);
    int bad = 0;
    if (nocc) {
        bad |= (unsigned long long)i > 0xFFFFFFFFull;
        O.trace[tp] = (uint32_t)i;   // index into the candidate list: the receiver adds the shard's first trace (no candidate
                                     // list on the exchange path: the index IS the shard-local trace index)
        if (O.base) O.base[tp] = G.s_ev_ts[se];
        if (!uniform) {
            bad |= (unsigned long long)(ep + (long long)v[2]) > 0xFFFFFFFFull;
            O.occ_off[tp] = (uint32_t)op;
            if (G.d_stage_occ) {
                const int64_t so = G.d_stage_occ[i];
                int64_t e = ep;
                for (uint32_t o = 0; o < nocc; ++o) {
                    O.ev_off[op + o] = (uint32_t)e;
                    e += G.s_occ_nev[so + o];
                }
            } else {
                O.ev_off[op] = (uint32_t)ep;
            }
        }
    }
    const unsigned my_ev = (unsigned)v[2];
    unsigned incl = my_ev;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
    }
    const unsigned wtot = __shfl_sync(0xffffffffu, incl, 31);
    const long long wbase = shfl_i64(ep, 0);
    for (unsigned f0 = 0; f0 < wtot; f0 += 32) {
        const unsigned f = f0 + lane;
        int lo = 0, hi = 31;
#pragma unroll
        for (int it = 0; it < 5; ++it) {
            const int mid = (lo + hi) >> 1;
            const unsigned vmid = __shfl_sync(0xffffffffu, incl, mid);
            if (vmid > f) hi = mid; else lo = mid + 1;
        }
        const int owner = lo & 31;
        const unsigned o_incl = __shfl_sync(0xffffffffu, incl, owner);
        const unsigned o_ev = __shfl_sync(0xffffffffu, my_ev, owner);
        const long long o_se = shfl_i64(se, owner);
        if (f < wtot) {
            const long long from = o_se + (long long)(f - (o_incl - o_ev));
            const long long to = wbase + f;
            const int32_t c_pos = __ldg(G.s_ev_pos + from);
            int32_t c_rank = 0, c_act = 0;
            long long c_ts = 0, c_base = 0;
            if (G.all_cols) {
                c_rank = __ldg(G.s_ev_rank + from);
                c_act = __ldg(G.s_ev_act + from);
                c_ts = __ldg(reinterpret_cast<const long long*>(G.s_ev_ts) + from);
                c_base = __ldg(reinterpret_cast<const long long*>(G.s_ev_ts) + o_se);
            }
            bad |= (unsigned)c_pos > 0xFFFFu;
            O.pos[to] = (uint16_t)c_pos;
            if (G.all_cols) {
                long long d = c_ts - c_base;
                if (O.seconds) {
                    bad |= d % 1000 != 0;
                    d /= 1000;
                }
                bad |= (unsigned)c_rank > 0xFFu || (unsigned)c_act > 0xFFFFu || d < -0x7fffffffll - 1 || d > 0x7fffffffll;
                O.rank[to] = (uint8_t)c_rank;
                O.act[to] = (uint16_t)c_act;
                O.delta[to] = (int32_t)d;
            }
        }
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(O.status, XST_RANGE);
}

// Header of the block: sizes from the request's counters, status, the tails of the offset sections, the error list.
__global__ void pack_header_kernel(const unsigned long long* counters, const int64_t* err_list, const int64_t* unsup_list, int unsup_slot,
                                   XHeader proto, XHeader* hdr, const __grid_constant__ PackSections O) {
    const int64_t n_occ = (int64_t)counters[0], n_ev = (int64_t)counters[1], n_tr = (int64_t)counters[6], n_err = (int64_t)counters[3];
    const int64_t n_unsup = (int64_t)counters[unsup_slot];
    if (threadIdx.x == 0) {
        int status = *O.status;
        if (n_unsup > XCHG_ERR_CAP || (long long)counters[7] > SIESTA_MAX_UNSUPPORTED) status |= XST_LIMITS;
        if (counters[5] > 0) status |= XST_STAGING;
        if (n_err > XCHG_ERR_CAP) status |= XST_ERRCAP;
        if (!proto.uniform_k && !(status & XST_STAGING)) {
            O.occ_off[n_tr] = (uint32_t)n_occ;
            O.ev_off[n_occ] = (uint32_t)n_ev;
        }
        proto.n_tr = n_tr;
        proto.n_occ = n_occ;
        proto.n_ev = n_ev;
        proto.n_err = n_err;
        proto.n_unsup = n_unsup;
        proto.n_emitted = (int64_t)counters[2];
        proto.status = status;
        *hdr = proto;
    }
    for (int64_t i = threadIdx.x; i < n_err && i < XCHG_ERR_CAP; i += blockDim.x) O.err[i] = err_list[i];
    for (int64_t i = threadIdx.x; i < n_unsup && i < XCHG_ERR_CAP; i += blockDim.x) O.unsup[i] = unsup_list[i];
}

// Would kernel K1-P take this request on a log with validated ids and an aligned activity column?  (siesta_evaluate_events
// decides with it whether a returnAll request can leave the timestamp column on the host: K1-P reads no timestamps to match,
// and only the few traces with more than one engine match are re-run on the staged kernel, which does.)
bool detect_nkp_eligible(const siesta_nfa* nfa, uint32_t flags, int32_t n_activities) {
    DevNfa dn;
    if (validate_nfa(nfa, flags, &dn) != SIESTA_OK || n_activities > 255 || std::getenv("SIESTA_K1_NO_NKP") != nullptr) return false;
    NkwProgram prog;
    if (nkw_build(dn, flags, &prog) == NKW_NONE) return false;
    std::vector<uint16_t> lut;
    int needs_ts = 0, n_positive = 0;
    build_lut(nfa, dn, n_activities, flags, lut, &needs_ts, &n_positive);
    std::vector<uint16_t> sigs;
    for (size_t a = 0; a < lut.size(); ++a) {
        const uint16_t sg = lut[a] & 0xFFu;
        if (sg && std::find(sigs.begin(), sigs.end(), sg) == sigs.end()) sigs.push_back(sg);
    }
    return !sigs.empty() && sigs.size() <= 7;
}

int detect_uniform_k(const siesta_nfa* nfa, uint32_t flags) {
    DevNfa dn;
    if (validate_nfa(nfa, flags, &dn) != SIESTA_OK || (flags & SIESTA_F_RETURN_ALL) || dn.any_kleene) return 0;
    int np = 0;
    for (int s = 0; s < nfa->n_states; ++s) np += nfa->states[s].kind != SIESTA_STATE_NEGATIVE;
    return std::max(1, np);
}

int64_t detect_pack_required_bytes(int64_t n, int64_t n_events_log, int uniform_k, bool all_cols, bool return_all) {
    const int64_t wide = std::min<int64_t>(n_events_log, n * 64);
    const int64_t cap_occ = return_all ? wide : n;
    const int64_t cap_ev = uniform_k ? n * uniform_k : wide;
    XHeader h;
    return (int64_t)pack_layout(std::max<int64_t>(n, 1), cap_occ, cap_ev, uniform_k, all_cols, &h);
}

void detect_pending_discard(DetectPending* q) { pending_discard(q); }
// Where the request's result sits in a larger one (shards of a multi-GPU log): may be set between the two halves, once
// the sizes of the shards before this one are known.  base.trace is added to the shard's first trace.
void detect_pending_set_base(DetectPending* q, RebaseOffsets base) {
    base.trace += q->log->first_trace;
    q->base = base;
}
// device time of the verification kernels alone (K1-P + staged re-run); valid once the request's stream has been waited for
float detect_pending_k1_ms(DetectPending* q) {
    float ms = 0.f;
    if (q && q->n > 0 && cudaEventElapsedTime(&ms, q->ev0, q->evd) != cudaSuccess) {
        cudaGetLastError();
        ms = 0.f;
    }
    return ms;
}

// Second half of a request on the exchange path: enqueues the placement into the exchange region and returns without
// waiting for the device.  The caller synchronises once all ranks' headers are in and then releases q
// (detect_pending_discard) - multi.cu.
int detect_device_pack_impl(DetectPending* q, const PackTarget& tgt) {
    Log* log = q->log;
    SIESTA_CUDA_OK(cudaSetDevice(log->ctx->device));
    cudaStream_t stream = q->stream;
    const int64_t n = q->n;
    const bool return_all = (q->flags & SIESTA_F_RETURN_ALL) != 0;
    const bool all_cols = (q->flags & SIESTA_F_NO_EVENT_COLUMNS) == 0;
    const DetectParams& P = q->P;
    if (q->d_cand) {
        set_error("exchange path: candidate lists are not supported (verify the whole shard)");
        return SIESTA_E_UNSUPPORTED;
    }
    XHeader proto;
    std::memset(&proto, 0, sizeof(proto));
    const size_t need = pack_layout(std::max<int64_t>(n, 1), P.cap_occ, P.cap_ev, q->uniform_k, all_cols, &proto);
    if ((int64_t)need > tgt.cap_bytes) {
        set_error("exchange region too small: " + std::to_string(need) + " bytes needed, " + std::to_string(tgt.cap_bytes) +
                  " available (siesta_exchange_required_bytes)");
        return SIESTA_E_NOMEM;
    }
    proto.seq = tgt.seq;
    proto.trace_base = q->base.trace;   // includes the shard's first trace
    proto.all_cols = all_cols ? 1 : 0;
    proto.seconds = (q->flags & SIESTA_F_EVT_POS) ? 0 : 1;
    proto.uniform_k = q->uniform_k;
    proto.slot_off = tgt.slot_off;
    proto.shard_traces = tgt.shard_traces;
    PackSections O;
    O.trace = reinterpret_cast<uint32_t*>(tgt.data + proto.o_trace);
    O.base = all_cols ? reinterpret_cast<int64_t*>(tgt.data + proto.o_base) : nullptr;
    O.occ_off = reinterpret_cast<uint32_t*>(tgt.data + proto.o_occ_off);
    O.ev_off = reinterpret_cast<uint32_t*>(tgt.data + proto.o_ev_off);
    O.pos = reinterpret_cast<uint16_t*>(tgt.data + proto.o_pos);
    O.rank = reinterpret_cast<uint8_t*>(tgt.data + proto.o_rank);
    O.act = reinterpret_cast<uint16_t*>(tgt.data + proto.o_act);
    O.delta = reinterpret_cast<int32_t*>(tgt.data + proto.o_delta);
    O.err = reinterpret_cast<int64_t*>(tgt.data + proto.o_err);
    O.unsup = reinterpret_cast<int64_t*>(tgt.data + proto.o_unsup);
    O.seconds = proto.seconds;
    O.status = reinterpret_cast<int*>(q->d_counters + 24);   // a zeroed word of the request's counter block
    if (n > 0) {
        GatherParams G;
        std::memset(&G, 0, sizeof(G));
        G.n = n;
        G.d_cnt = P.d_cnt;
        G.d_stage = P.d_stage;
        G.d_stage_occ = return_all ? P.d_stage_occ : nullptr;
        G.n_blk = (int64_t)q->n_blk;
        G.blk = q->d_blk;
        G.n_chunks = (int64_t)((q->n_blk + 1023) / 1024);
        G.top = q->d_top;
        G.s_occ_nev = P.s_occ_nev;
        G.s_ev_pos = P.s_ev_pos;
        G.s_ev_rank = P.s_ev_rank;
        G.s_ev_act = P.s_ev_act;
        G.s_ev_ts = P.s_ev_ts;
        G.all_cols = all_cols ? 1 : 0;
        G.tile_words = q->tile_words;
        G.n_tiles = q->n_tiles;
        G.fix_ev = q->fix_ev;
        scan_chunks_kernel<<<(unsigned)G.n_chunks, SC, 0, stream>>>(G.blk, G.n_blk, G.top, G.n_chunks);
        SIESTA_LAUNCHED();
        scan_top_kernel<<<1, SC, 0, stream>>>(G.top, G.n_chunks);
        SIESTA_LAUNCHED();
        if (q->tile_words)
            gather_uniform_kernel<true><<<(unsigned)((G.n_blk + GT / 32 - 1) / (GT / 32)), GT, 0, stream>>>(G, O, q->uniform_k);
        else
            gather_packed_kernel<<<(unsigned)G.n_blk, GT, 0, stream>>>(G, O, q->uniform_k ? 1 : 0);
        SIESTA_LAUNCHED();
    }
    pack_header_kernel<<<1, 256, 0, stream>>>(q->d_counters, q->d_err, q->d_unsup, q->unsup_slot, proto, tgt.hdr, O);
    SIESTA_LAUNCHED();
    SIESTA_CUDA_OK(cudaGetLastError());
    return SIESTA_OK;
}

int detect_device_impl(Log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand, uint32_t flags,
                       cudaStream_t stream, RebaseOffsets base, siesta_dev_matches* out) {
    std::memset(out, 0, sizeof(*out));
    DetectPending* q = nullptr;
    const int rc = detect_device_begin_impl(log, nfa, d_cand, n_cand, flags, stream, base, &q);
    if (rc != SIESTA_OK) return rc;
    return detect_device_finish_impl(q, out);
}

}  // namespace siesta

extern "C" int siesta_detect_device_begin(siesta_log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand,
                                          uint32_t flags, void* stream, siesta_detect_pending** out) {
    if (!log || !nfa || !out || (d_cand && n_cand < 0)) {
        siesta::set_error("siesta_detect_device_begin: null argument");
        return SIESTA_E_INVALID;
    }
    siesta::DetectPending* q = nullptr;
    const int rc = siesta::detect_device_begin_impl(reinterpret_cast<siesta::Log*>(log), nfa, d_cand, n_cand, flags,
                                                    reinterpret_cast<cudaStream_t>(stream), siesta::RebaseOffsets{0, 0, 0}, &q);
    *out = reinterpret_cast<siesta_detect_pending*>(q);
    return rc;
}

extern "C" int siesta_detect_device_finish(siesta_detect_pending* pending, siesta_dev_matches* out) {
    if (!pending || !out) {
        siesta::set_error("siesta_detect_device_finish: null argument");
        return SIESTA_E_INVALID;
    }
    return siesta::detect_device_finish_impl(reinterpret_cast<siesta::DetectPending*>(pending), out);
}

extern "C" int siesta_detect_device(siesta_log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand,
                                    uint32_t flags, void* stream, siesta_dev_matches* out) {
    if (!log || !nfa || !out || (d_cand && n_cand < 0)) {
        siesta::set_error("siesta_detect_device: null argument");
        return SIESTA_E_INVALID;
    }
    return siesta::detect_device_impl(reinterpret_cast<siesta::Log*>(log), nfa, d_cand, n_cand, flags,
                                      reinterpret_cast<cudaStream_t>(stream), siesta::RebaseOffsets{0, 0, 0}, out);
}

extern "C" void siesta_dev_matches_free(siesta_dev_matches* m) {
    if (!m || !m->impl) return;
    siesta::DevMatchesImpl* impl = reinterpret_cast<siesta::DevMatchesImpl*>(m->impl);
    siesta::dev_arena_free(impl->owner, impl->block);   // the caller is done with the result: its block serves the next request
    delete impl;
    m->impl = nullptr;
}
