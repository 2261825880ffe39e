/*
 * siesta_gpu.h — C-ABI of the B200-native SIESTA pattern-query hot path.
 *
 * This is the drop-in boundary a thin JNI class binds (see INTEGRATION.md).
 * The reference (siesta-tool/SequenceDetectionQueryExecutor) is pure Java and
 * has no FFI of its own; every entry point below names the Java seam it
 * replaces (paths relative to the reference's
 * src/main/java/com/datalab/siesta/queryprocessor/, "S/" =
 * src/main/java/edu/umass/cs/sase/).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, little-endian, no exceptions.
 *   - Every int function returns 0 on success or a negative SIESTA_E_* code;
 *     siesta_last_error() returns a thread-local message for the last failure.
 *   - Inputs are borrowed for the duration of the call.  The library owns all
 *     device memory and every result object it returns (free with the
 *     matching *_free).
 *   - Activity names and trace ids are mapped to dense integers by the
 *     caller.  Names must be folded case-insensitively first because the
 *     engine compares types with equalsIgnoreCase (S/query/State.java:135,
 *     S/query/AdditionalState.java:45-52).
 *   - There is no CPU fallback: every compute entry point fails with
 *     SIESTA_E_CUDA when no sm_100 device is usable.
 */
#ifndef SIESTA_GPU_H
#define SIESTA_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ errors */
#define SIESTA_OK 0
#define SIESTA_E_INVALID (-1)     /* bad argument / malformed NFA                */
#define SIESTA_E_CUDA (-2)        /* CUDA runtime failure, or no device          */
#define SIESTA_E_UNSUPPORTED (-3) /* NFA shape / flag combination the GPU engine does not accept */
#define SIESTA_E_NOMEM (-4)
#define SIESTA_E_REFERENCE_THROWS (-5) /* the Java engine would throw (see n_ref_errors) */

const char* siesta_last_error(void);

/* --------------------------------------------------------------------- NFA */
/* State kinds: ComplexPattern.getStatesWithoutConstraints (model/Patterns/
 * ComplexPattern.java:216-272): "_"->normal, "+"->kleeneClosure,
 * "*"->kleeneClosure*, "!"->negative, "||"->or. */
#define SIESTA_STATE_NORMAL 0
#define SIESTA_STATE_KLEENE_PLUS 1
#define SIESTA_STATE_KLEENE_STAR 2
#define SIESTA_STATE_NEGATIVE 3
#define SIESTA_STATE_OR 4

#define SIESTA_ATTR_POSITION 0
#define SIESTA_ATTR_TIMESTAMP 1
#define SIESTA_OP_LE 0 /* "within"  -> attr <= $ref.attr + c (SIESTAPattern.java:136,142) */
#define SIESTA_OP_GE 1 /* otherwise -> attr >= $ref.attr + c (SIESTAPattern.java:138,144) */

#define SIESTA_MAX_STATES 8
#define SIESTA_MAX_OR_TYPES 8
#define SIESTA_MAX_PREDS 4

/* One predicate " attr <=|>= $<ref_state+1>.attr + constant "
 * (model/Patterns/SIESTAPattern.java:131-149).  SIESTA attaches the same list
 * to the begin edge and, for both Kleene kinds, to the take edge; never to
 * the proceed edge (ComplexPattern.java:200-208), so one list per state is
 * the complete description. */
typedef struct siesta_pred {
    int32_t attr;      /* SIESTA_ATTR_*                         */
    int32_t op;        /* SIESTA_OP_*                           */
    int32_t ref_state; /* 0-based index of the referenced state */
    int32_t reserved;
    int64_t constant;  /* >= 0; seconds for timestamp           */
} siesta_pred;

typedef struct siesta_state {
    int32_t kind;    /* SIESTA_STATE_*                                     */
    int32_t n_types; /* 1, or >1 for an "or" state                         */
    int32_t types[SIESTA_MAX_OR_TYPES]; /* dense activity ids              */
    int32_t n_preds;
    int32_t reserved;
    siesta_pred preds[SIESTA_MAX_PREDS];
} siesta_state;

typedef struct siesta_nfa {
    int32_t n_states;
    int32_t reserved;
    siesta_state states[SIESTA_MAX_STATES];
} siesta_nfa;

/* ------------------------------------------------------- pattern compiler */
/* Replaces ComplexPattern.getNfa / getNfaWithoutConstraints
 * (ComplexPattern.java:194-214, 274-283), SimplePattern.getNfa
 * (SimplePattern.java:96-104) and SIESTAPattern.generatePredicates
 * (SIESTAPattern.java:131-149).  Host only. */
#define SIESTA_SYM_NORMAL 0 /* "_" (and "") */
#define SIESTA_SYM_PLUS 1   /* "+"  */
#define SIESTA_SYM_STAR 2   /* "*"  */
#define SIESTA_SYM_NOT 3    /* "!"  */
#define SIESTA_SYM_OR 4     /* "||" */

typedef struct siesta_event_symbol {
    int32_t activity; /* dense activity id                    */
    int32_t position; /* EventSymbol.position in the pattern  */
    int32_t symbol;   /* SIESTA_SYM_*                         */
} siesta_event_symbol;

#define SIESTA_CONSTRAINT_GAP 0
#define SIESTA_CONSTRAINT_TIME 1
#define SIESTA_METHOD_WITHIN 0
#define SIESTA_METHOD_ATLEAST 1
#define SIESTA_GRAN_SECONDS 0
#define SIESTA_GRAN_MINUTES 1
#define SIESTA_GRAN_HOURS 2

typedef struct siesta_constraint {
    int32_t pos_a, pos_b; /* state indices, pos_a < pos_b (Constraint.java:98-100) */
    int32_t kind;         /* SIESTA_CONSTRAINT_*                                    */
    int32_t method;       /* SIESTA_METHOD_*                                        */
    int64_t value;
    int32_t granularity;  /* SIESTA_GRAN_* (time constraints only)                  */
    int32_t reserved;
} siesta_constraint;

int siesta_pattern_compile(const siesta_event_symbol* symbols, int32_t n_symbols,
                           const siesta_constraint* constraints, int32_t n_constraints,
                           int32_t only_appearances, siesta_nfa* out);

/* Replaces ComplexPattern.extractPairsForPatternDetection(fromOrTillSet) (ComplexPattern.java:75-128) and
 * SIESTAPattern.extractPairsForPatternDetection (SIESTAPattern.java:34-69): per OR-expansion of the pattern
 * (splitWithOr, ComplexPattern.java:130-171) the "true" pairs (every ordered pair of "_" / "+" events: a trace must
 * hold all of them) and "all" pairs (true pairs + the pairs fetched for "*", "!", self pairs).  Pair sets are sets of
 * (a, b) activity ids (EventPair equality is by name, EventPair.java:65-81), returned sorted; expansion x owns
 * true_a/b[true_off[x] .. true_off[x+1]) and all_a/b[all_off[x] .. all_off[x+1]).  Returns
 * SIESTA_E_REFERENCE_THROWS for the patterns on which the Java code loops forever (ComplexPattern.java:108-113).
 * Host only. */
int siesta_pattern_extract_pairs(const siesta_event_symbol* symbols, int32_t n_symbols,
                                 const siesta_constraint* constraints, int32_t n_constraints, int32_t from_or_till_set,
                                 int32_t cap_expansions, int32_t cap_pairs, int32_t* n_expansions,
                                 int32_t* true_off /* [cap_expansions + 1] */, int32_t* true_a, int32_t* true_b,
                                 int32_t* all_off /* [cap_expansions + 1] */, int32_t* all_a, int32_t* all_b);

/* ------------------------------------------------------------ ctx and log */
typedef struct siesta_ctx siesta_ctx;
typedef struct siesta_log siesta_log;

/* One ctx per (process, device).  Multi-GPU = one ctx per GPU; the traces
 * shard by contiguous trace range and the exchange step (match-list
 * all-gather, count all-reduce) is siesta_exchange_* (below). */
int siesta_init(int32_t device_id, siesta_ctx** out);
void siesta_shutdown(siesta_ctx* ctx);

/* CSR event log: trace_off[T+1] (int64), act[E] (int32 dense activity id),
 * ts_ms[E] (int64 epoch milliseconds, sorted inside each trace).  Replaces the
 * Map<String, List<Event>> the reference materialises per request
 * (SaseConnection/SaseConnector.java:48-51, storage/repositories/
 * SparkDatabaseRepository.java:94-107).  Copies host -> device. */
int siesta_log_load(siesta_ctx* ctx, const int64_t* trace_off, const int32_t* act,
                    const int64_t* ts_ms, int64_t n_traces, int64_t n_events,
                    int32_t n_activities, siesta_log** out);
/* Same, over device memory the caller owns and keeps alive (torch tensors). */
int siesta_log_wrap_device(siesta_ctx* ctx, const int64_t* d_trace_off, const int32_t* d_act,
                           const int64_t* d_ts_ms, int64_t n_traces, int64_t n_events,
                           int32_t n_activities, int32_t max_trace_len, siesta_log** out);
/* Multi-GPU: this log is the shard [first_trace, first_trace + n_traces) of a larger log.  Every trace index the
 * library RETURNS for it (trace_idx, err_trace_idx) is then global; candidate lists stay local to the shard. */
void siesta_log_set_first_trace(siesta_log* log, int64_t first_trace);
/* Multi-GPU, block-cyclic shard: the log is cut into n_blocks * world blocks of consecutive traces and rank r holds
 * blocks r, world + r, 2 world + r, ... back to back.  Block b of THIS shard = its local traces
 * [local_first[b], local_first[b + 1]) = the global traces starting at global_first[b] (local_first[0] = 0,
 * local_first[n_blocks] = the shard's trace count, 1 <= n_blocks <= SIESTA_MAX_BLOCKS, the same on every rank).
 * siesta_detect_allgather then runs block by block: while block b + 1 is verified, block b of every rank is already
 * pulled over NVLink and decoded at its place in the joined list, which stays in global trace order (block 0 of rank
 * 0, 1, ..., block 1 of rank 0, ...).  Other entry points keep reporting first_trace + local index for such a log.
 * n_blocks = 0 clears the declaration. */
#define SIESTA_MAX_BLOCKS 16
int siesta_log_set_blocks(siesta_log* log, int32_t n_blocks, const int64_t* local_first, const int64_t* global_first);
void siesta_log_free(siesta_log* log);
int64_t siesta_log_n_traces(const siesta_log* log);
int64_t siesta_log_n_events(const siesta_log* log);

/* ---------------------------------------------------- derived logs (device) */
/* Trace.filter(from, till) (model/DBModel/Trace.java:25-29; the same test in SparkDatabaseRepository.addFilterIds
 * :204-218 and Utils.evaluateEvent, model/Utils/Utils.java:67-79) over a resident log, on the device: a new resident
 * log that holds, per trace, the events with from_ms <= timestamp <= till_ms (a bound counts only if its has_* flag is
 * set).  The reference filters the event list BEFORE numbering it, so positions in the derived log are ranks among
 * the surviving events; siesta_log_source_events gives each event's index in the source log.  Traces keep their
 * indices (a trace may become empty).  Free with siesta_log_free. */
int siesta_log_filter_time(siesta_log* log, int64_t from_ms, int32_t has_from, int64_t till_ms, int32_t has_till,
                           siesta_log** out);
/* The streams of /detection over groups of traces (SparkDatabaseRepository.querySingleTableGroups :307-336, evaluated
 * by SaseConnector.evaluateGroups, SaseConnector.java:85-110 = siesta_detect on the log returned here): group g lists
 * the traces group_traces[group_off[g] .. group_off[g+1]); a trace belongs to the FIRST group that lists it; a group's
 * stream is the events of its traces merged by timestamp (ties: order of the trace in the group's list, then position
 * - the reference's order of ties is undefined); a group whose events do not cover all n_types event types of the
 * query (<= 64) is dropped.  Trace i of the new log is the i-th kept group, group_ids[i] its 1-based number as the
 * reference reports it (:317); group_ids must hold n_groups entries.  Traces must be sorted by timestamp. */
int siesta_log_group(siesta_log* log, const int64_t* group_off, const int64_t* group_traces, int32_t n_groups,
                     const int32_t* types, int32_t n_types, siesta_log** out, int32_t* group_ids, int32_t* n_kept);
/* Derived logs only: out[e] = index in the SOURCE log of event e (host array of siesta_log_n_events entries). */
int siesta_log_source_events(siesta_log* log, int64_t* out);

/* ------------------------------------------------------ growing a resident log */
/* A new resident log = `log` with a batch of events appended, rebuilt on the device.  The batch is a CSR over the
 * traces it touches: trace_idx[n_listed] strictly ascending LOCAL trace indices in [0, T + n_new_traces),
 * batch_off[n_listed + 1] (batch_off[0] = 0, non-decreasing), act / ts_ms[batch_off[n_listed]].  The events of listed
 * trace i go after the existing events of trace trace_idx[i], in the given order.  Indices >= T are new traces; new
 * traces that are not listed are empty.  n_activities >= the log's (the dictionary only grows).  Activity ids outside
 * [0, n_activities) are accepted as siesta_log_load accepts them; timestamps must stay sorted inside each trace (not
 * checked, as in siesta_log_load).  The new log keeps the log's first_trace and owns its memory.
 * `log` itself is NOT modified and stays valid: requests may keep running on it, and the caller frees it
 * (siesta_log_free) when none does.  Peak device memory: the old log + the new log + the batch staging.
 * SIESTA_E_INVALID (nothing changed, *out untouched): a null argument, trace indices not strictly ascending or out of
 * range, n_new_traces < 0, malformed batch_off, n_activities below the log's, a derived log (siesta_log_filter_time /
 * siesta_log_group) or a block-cyclic shard (siesta_log_set_blocks).  SIESTA_E_NOMEM: an allocation failed; the old
 * log is intact.  *kernel_ms (may be NULL) = device time of the rebuild (CUDA events; excludes the host -> device copy
 * of the batch).  The events are recorded on the context's stream, so work that other threads enqueue on the same
 * context during the call is counted too; the time is the rebuild's alone only when nothing else runs on the context. */
int siesta_log_append(siesta_log* log, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                      const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces, int32_t n_activities,
                      siesta_log** out, double* kernel_ms);
/* Host copy of traces [t0, t1) of a resident log: trace_off[t1 - t0 + 1] (offsets into the log's event columns, as
 * stored), act / ts_ms[trace_off[t1-t0] - trace_off[0]] (both NULL: offsets only). */
int siesta_log_read(siesta_log* log, int64_t t0, int64_t t1, int64_t* trace_off, int32_t* act, int64_t* ts_ms);

/* -------------------------------------------------------------- detection */
/* flags */
#define SIESTA_F_RETURN_ALL 1u       /* Occurrences.clearOccurrences(true) (model/Occurrences.java:58-89) */
#define SIESTA_F_ONLY_APPEARANCES 2u /* ignore predicates (SaseConnector.java:156-158)                     */
#define SIESTA_F_MODE_HEAD 4u        /* keep Engine.createNewRun's trailing block (S/engine/Engine.java:983-996);
                                        default is the mode the reference's own tests pin (DESIGN.md)      */
#define SIESTA_F_EVT_POS 8u          /* events are EventPos: id = true position, timestamp = list index
                                        (model/Utils/Utils.java:59-62); default EventTs/EventBoth:
                                        id = list index, timestamp = (t - t0)/1000 s (Utils.java:51-58)    */
#define SIESTA_F_NO_EVENT_COLUMNS 16u /* return only trace_idx/occ_off/ev_off/ev_pos                       */
#define SIESTA_F_COUNT_MATCHES 32u    /* also report the exact number of engine matches before selection
                                         (n_matches_emitted); without it the engine may drop runs that can
                                         never yield the selected occurrence and reports -1              */
#define SIESTA_F_LITERAL_RUNS 64u     /* keep the run list exactly as the Java engine does (no inert-run pruning,
                                         no dominated-run merging); same output, slower; for audits and tests  */

/* Result of SaseConnector.evaluate + Occurrences.clearOccurrences, CSR-shaped.
 * Host memory owned by the library. */
typedef struct siesta_matches {
    int64_t n_traces;          /* traces with >= 1 match                             */
    int64_t n_occurrences;     /* selected occurrences over all traces               */
    int64_t n_events;          /* events over all selected occurrences               */
    int64_t n_matches_emitted; /* engine matches before selection (Profiling.numberOfMatches); -1 unless
                                  SIESTA_F_COUNT_MATCHES, SIESTA_F_RETURN_ALL or SIESTA_F_LITERAL_RUNS      */
    int64_t n_ref_errors;      /* traces on which the Java engine would throw        */
    int64_t* trace_idx;        /* [n_traces] ascending                               */
    int64_t* occ_off;          /* [n_traces+1] -> occurrence range of a trace        */
    int64_t* ev_off;           /* [n_occurrences+1] -> event range of an occurrence  */
    int32_t* ev_pos;           /* [n_events] index of the event inside its trace     */
    int32_t* ev_rank;          /* [n_events] index in the list filtered to the pattern's types */
    int32_t* ev_act;           /* [n_events] activity id                             */
    int64_t* ev_ts_ms;         /* [n_events] SaseEvent.getEventBoth timestamp: rel_s*1000 + t0 (SaseEvent.java:94-106) */
    int64_t* err_trace_idx;    /* [n_ref_errors] ascending                           */
    double kernel_ms;          /* device time of all kernels of the call (CUDA events) */
    double detect_ms;          /* device time of the verification kernel K1 alone      */
    /* Traces beyond the GPU engine's per-trace limits: for a pattern WITH a Kleene state, more than 64 pattern-relevant
     * events, 1024 live runs or 65 536 events (patterns without one are evaluated on traces of any length, kernel K1-L,
     * and never list a trace).  The reference has no such limit (S/engine/Engine.java:207-224), so the request does NOT fail for them:
     * every other trace is answered and these are listed (ascending) for the caller to evaluate elsewhere - the JNI
     * shim hands them to the reference's own engine (INTEGRATION.md).  More than SIESTA_MAX_UNSUPPORTED of them fail
     * the call with SIESTA_E_UNSUPPORTED. */
    int64_t n_unsupported;
    int64_t* unsupported_trace_idx; /* [n_unsupported] */
} siesta_matches;
#define SIESTA_MAX_UNSUPPORTED 65536

/* Replaces SaseConnector.evaluate(pattern, events, onlyAppearances) followed by
 * occurrences.forEach(clearOccurrences(returnAll))
 * (SaseConnector.java:48-76; QueryPlanPatternDetection.java:121-122).
 * cand = NULL verifies every trace of the log; otherwise cand[n_cand] are
 * ascending trace indices (the output of siesta_intersect).
 * Re-entrant: concurrent calls on one log from different threads are safe. */
int siesta_detect(siesta_log* log, const siesta_nfa* nfa, const int64_t* cand, int64_t n_cand,
                  uint32_t flags, siesta_matches** out);
void siesta_matches_free(siesta_matches* m);

/* Literal SaseConnector.evaluate signature: the caller hands the events of
 * this request (host CSR); equals log_load + detect + log_free, in chunks that
 * overlap the host link with the kernels.  When no predicate of the pattern
 * reads relative seconds and ts_ms lies in page-locked host memory
 * (cudaHostAlloc / cudaHostRegister), the timestamp column is not copied: the
 * kernels read the reported events' timestamps in place (4 B/event on the
 * link instead of 12).  Pageable columns are copied; same results either way. */
int siesta_evaluate_events(siesta_ctx* ctx, const int64_t* trace_off, const int32_t* act,
                           const int64_t* ts_ms, int64_t n_traces, int64_t n_events,
                           int32_t n_activities, const siesta_nfa* nfa, uint32_t flags,
                           siesta_matches** out);

/* The same request with the activity column as ONE BYTE per event (n_activities
 * <= 256).  siesta_evaluate_events runs at the speed of the host link and the
 * activity column is what crosses it, so the caller's serialiser - the JNI shim
 * that flattens Map<String, List<Event>> (SaseConnector.java:48) into direct
 * buffers - writes the dictionary id into a byte: 1 B/event on the link instead
 * of 4.  The device widens each chunk to the int32 column the kernels read.
 * Same results as siesta_evaluate_events on the widened column. */
int siesta_evaluate_events_act8(siesta_ctx* ctx, const int64_t* trace_off, const uint8_t* act8,
                                const int64_t* ts_ms, int64_t n_traces, int64_t n_events,
                                int32_t n_activities, const siesta_nfa* nfa, uint32_t flags,
                                siesta_matches** out);

/* Device-level variant for callers that consume the result on the device: results stay in HBM.
 * All pointers are device pointers owned by the library until
 * siesta_dev_matches_free; `stream` is a cudaStream_t (NULL = the ctx stream). */
typedef struct siesta_dev_matches {
    int64_t n_traces, n_occurrences, n_events, n_matches_emitted, n_ref_errors;
    int64_t* d_trace_idx;
    int64_t* d_occ_off;
    int64_t* d_ev_off;
    int32_t* d_ev_pos;
    int32_t* d_ev_rank;
    int32_t* d_ev_act;
    int64_t* d_ev_ts_ms;
    int64_t* d_err_trace_idx;
    double kernel_ms;
    double detect_ms;
    /* all eight arrays above live in ONE device allocation [d_block, d_block + block_bytes), each at a 256-byte
     * aligned offset, in the order trace_idx, occ_off, ev_off, ev_pos, err_trace_idx, ev_rank, ev_act, ev_ts_ms */
    void* d_block;
    int64_t block_bytes;
    void* impl;
    int64_t n_unsupported;            /* as in siesta_matches; the ninth array of the block */
    int64_t* d_unsupported_trace_idx;
} siesta_dev_matches;

int siesta_detect_device(siesta_log* log, const siesta_nfa* nfa, const int64_t* d_cand,
                         int64_t n_cand, uint32_t flags, void* stream, siesta_dev_matches* out);
/* The same request in two halves, for callers that keep several requests in flight (the reference serves concurrent
 * requests; the multi-GPU exchange of request i then overlaps the scan of request i + 1): _begin enqueues the
 * verification kernels and returns without waiting for the device; _finish waits for them, allocates the result,
 * places it and fills `out` exactly as siesta_detect_device does.  _finish consumes `pending` whatever it returns; every
 * _begin must be followed by exactly one _finish (also to release the request after an error elsewhere).  `nfa` and
 * `d_cand` are borrowed until _finish returns. */
typedef struct siesta_detect_pending siesta_detect_pending;
int siesta_detect_device_begin(siesta_log* log, const siesta_nfa* nfa, const int64_t* d_cand, int64_t n_cand,
                               uint32_t flags, void* stream, siesta_detect_pending** out);
int siesta_detect_device_finish(siesta_detect_pending* pending, siesta_dev_matches* out);
void siesta_dev_matches_free(siesta_dev_matches* m);

/* ------------------------------------------------------- multi-GPU exchange */
/* Traces are independent, so a log shards by contiguous trace range, one shard per GPU (siesta_log_set_first_trace),
 * and every kernel of this library runs on every shard unchanged.  The results are joined on the devices, over NVLink
 * peer memory: the match lists by an all-gather (siesta_detect_allgather), the count arrays of /declare, /stats and
 * /explore by an all-reduce (siesta_exchange_allreduce_i64).  The reference has no counterpart (one JVM, Spark
 * local[*]); the loop that the shards split is SaseConnector.evaluate's loop over all candidate traces
 * (SaseConnection/SaseConnector.java:51-74) behind QueryPlanPatternDetection.execute (model/Queries/QueryPlans/
 * Detection/QueryPlanPatternDetection.java:106-131).
 *
 * One siesta_exchange per rank (GPU).  Every rank owns a device region that all its peers map:
 *   one process per GPU (torchrun, one JVM per GPU): siesta_exchange_export gives a 64-byte handle (cudaIpcMemHandle_t)
 *     that the host layer hands to the other ranks by any means; each rank calls siesta_exchange_import once per peer;
 *   one process driving all GPUs (a single JVM): siesta_exchange_connect_local once per ordered pair (peer access).
 * Collective calls (siesta_detect_allgather, siesta_exchange_allreduce_i64) must be issued by every rank in the same
 * order.  Sizes travel in-band and every device-side wait is bounded: a missing peer fails the call (SIESTA_E_CUDA)
 * after 20 s instead of hanging the GPU.  csrc/multi.cu describes the protocol and the compact block format. */
typedef struct siesta_exchange siesta_exchange;
#define SIESTA_EXCHANGE_HANDLE_BYTES 64
int siesta_exchange_create(siesta_ctx* ctx, int32_t world, int32_t rank, int64_t capacity_bytes, siesta_exchange** out);
int siesta_exchange_export(siesta_exchange* x, void* handle_out /* SIESTA_EXCHANGE_HANDLE_BYTES */);
int siesta_exchange_import(siesta_exchange* x, int32_t peer_rank, const void* handle);
int siesta_exchange_connect_local(siesta_exchange* x, int32_t peer_rank, siesta_exchange* peer);
void siesta_exchange_free(siesta_exchange* x);
/* Bytes of exchange region a /detection request on this shard needs (worst case of its compact block): the host
 * layer creates the exchanges with the maximum over the ranks. */
int64_t siesta_exchange_required_bytes(siesta_log* log, const siesta_nfa* nfa, uint32_t flags);

typedef struct siesta_exchange_stats {
    int64_t local_traces, local_occurrences, local_events; /* this rank's share of the joined list              */
    int64_t pulled_bytes;                                  /* bytes read from the peers' regions over NVLink      */
    double k1_ms;    /* the verification kernels alone (device time)                                              */
    double scan_ms;  /* verification + placement of this rank's block (device time)                               */
    double wait_ms;  /* announce + wait for the slowest rank + fetch of the headers                               */
    double pull_ms;  /* pull + decode of all blocks into the joined columns                                       */
    double host_gap_ms; /* between the two: the host reads the sizes and allocates the joined result              */
    /* block-pipelined requests (siesta_log_set_blocks): scan_ms spans all blocks, pull_ms is what the join adds behind
     * the last block's announcement (wait_ms and host_gap_ms are 0), join_ms the span of the join stream */
    double join_ms;
    int32_t n_blocks; /* blocks the shard was processed in (1 = contiguous shard)                                 */
    int32_t eager;    /* 1: joined columns allocated for the worst case up front and filled block by block         */
} siesta_exchange_stats;

/* siesta_detect_device over this rank's shard FOLLOWED BY the all-gather: `out` holds the match list of ALL ranks in
 * trace order (global trace indices), in the library's standard columns, on this rank's device.  The verification
 * kernels place their result directly into the exchange region as a compact block whose header carries the sizes;
 * one kernel then pulls every peer's block over NVLink and decodes it at its place in the joined list.  The host
 * waits twice (sizes of the first blocks; end of the request).  An error on any rank fails the call on every rank.
 * Block-cyclic shards (siesta_log_set_blocks): the scan, the placement and the announcement of block b + 1 run on one
 * stream while a second stream waits for block b of every rank, pulls and decodes it - the join overlaps the scan.
 * When every match has the same shape (no Kleene state, first-largest occurrence) the joined columns are allocated
 * for the worst case up front (every trace of every shard matches; the shard sizes travel in the headers) and filled
 * block by block at running offsets computed on the device: `out`'s arrays are then compact, but they sit at
 * capacity-based offsets inside d_block.  Other requests on a blocked log decode after the last block (exact
 * allocation), so only their pulls' latency is hidden.  SIESTA_XCHG_EAGER_MAX_BYTES (default 24 GiB) bounds the
 * worst-case allocation; above it the request decodes after the last block. */
int siesta_detect_allgather(siesta_log* log, const siesta_nfa* nfa, uint32_t flags, siesta_exchange* x,
                            siesta_dev_matches* out, siesta_exchange_stats* stats /* may be NULL */);

#define SIESTA_REDUCE_SUM 0
#define SIESTA_REDUCE_MIN 1
#define SIESTA_REDUCE_MAX 2
/* In-place all-reduce of a device array of int64 (the packed counts of siesta_declare_counts_device, the records of
 * siesta_pair_stats_device, the completions of /explore): every rank ends with op over all ranks, combined in rank
 * order (deterministic).  `stream` = the cudaStream_t that produced d_buf (NULL = the ctx stream); returns when done. */
int siesta_exchange_allreduce_i64(siesta_exchange* x, int64_t* d_buf, int64_t n, int32_t op, void* stream);

/* One process driving all GPUs (the reference is ONE JVM): a context and an exchange per device, connected through
 * peer access; a host CSR log sharded by contiguous trace range balanced by event count; every request entry point
 * runs all shards at once, one host thread per device.  /detection results are joined on the HOST (each device copies
 * its columns into its slice of one pinned block: all host links in parallel), counts are all-reduced on the devices.
 * device_ids may name a device more than once (several shards on one GPU: tests). */
typedef struct siesta_multi siesta_multi;
typedef struct siesta_multi_log siesta_multi_log;
int siesta_multi_init(const int32_t* device_ids, int32_t n_dev, siesta_multi** out);
void siesta_multi_shutdown(siesta_multi* m);
int32_t siesta_multi_n_devices(const siesta_multi* m);
int siesta_multi_log_load(siesta_multi* m, const int64_t* trace_off, const int32_t* act, const int64_t* ts_ms,
                          int64_t n_traces, int64_t n_events, int32_t n_activities, siesta_multi_log** out);
void siesta_multi_log_free(siesta_multi_log* log);
siesta_log* siesta_multi_log_shard(siesta_multi_log* log, int32_t shard); /* borrowed: any single-GPU call on one shard */
/* siesta_log_append over a sharded log.  trace_idx are GLOBAL.  New traces go to the last shard (shards are not
 * rebalanced).  Every shard is rebuilt on its device from its own host thread; a shard with no listed trace is
 * copied, so the new multi log owns all of its shards.  The old multi log stays valid and unchanged; if one shard
 * fails, the shards already built are freed and the error is returned. */
int siesta_multi_log_append(siesta_multi_log* log, const int64_t* trace_idx, const int64_t* batch_off, int64_t n_listed,
                            const int32_t* act, const int64_t* ts_ms, int64_t n_new_traces, int32_t n_activities,
                            siesta_multi_log** out);
/* = siesta_detect(whole log, nfa, NULL, 0, flags): SaseConnector.evaluate + clearOccurrences
 * (SaseConnection/SaseConnector.java:48-76), global trace indices, trace order. */
int siesta_multi_detect(siesta_multi_log* log, const siesta_nfa* nfa, uint32_t flags, siesta_matches** out);
/* = siesta_declare_counts(whole log): kernel K3 per shard + one sum all-reduce over the exchange. */
int siesta_multi_declare_counts(siesta_multi_log* log, int32_t k_cap, int64_t* out, double* kernel_ms);
/* = siesta_declare_counts_refresh over all shards (new_log = siesta_multi_log_append(old_log, ...)): trace_idx are GLOBAL
 * and split as the append splits them (new traces on the last shard).  Every shard is checked before anything is
 * counted; each computes its delta, one sum all-reduce joins them and one merge adds them to old_counts.  The count array
 * must fit the exchange region, as for siesta_multi_declare_counts.  Same refusals and fallback. */
int siesta_multi_declare_counts_refresh(siesta_multi_log* old_log, siesta_multi_log* new_log, const int64_t* trace_idx,
                                        int64_t n_listed, int32_t k_cap, const int64_t* old_counts, int64_t* out,
                                        double* kernel_ms);
/* siesta_why_not_match (below) over all shards: cand = ascending GLOBAL trace indices (NULL: every trace); every
 * device answers its own candidates, the answers are concatenated in trace order. */
struct siesta_wnm_constraint;
struct siesta_almost_matches;
int siesta_multi_why_not_match(siesta_multi_log* log, const int32_t* pattern_activities, int32_t n_pattern,
                               const struct siesta_wnm_constraint* constraints, int32_t n_constraints,
                               int32_t uncertainty, int32_t step, int32_t k, const int64_t* cand, int64_t n_cand,
                               uint32_t flags, struct siesta_almost_matches** out);

/* ------------------------------------------------- pair index + intersection */
/* Kernel K2.  Replaces SparkDatabaseRepository.getCommonIds (storage/repositories/
 * SparkDatabaseRepository.java:160-178): the traces that contain ALL true pairs = the intersection of the
 * per-pair posting lists (ascending, duplicate-free dense trace indices). */
typedef struct siesta_index siesta_index;

/* Posting lists produced elsewhere (index.parquet rows of S3Connector.getAllEventPairs :236-292, mapped to dense
 * trace indices and sorted by the caller): list p = trace_idx[post_off[p] .. post_off[p+1]). */
int siesta_index_load(siesta_log* log, int32_t n_pairs, const int32_t* pair_a, const int32_t* pair_b,
                      const int64_t* post_off, const int64_t* trace_idx, siesta_index** out);
/* Posting lists derived on the GPU from the resident CSR log under the SeqTable view: a trace is listed under
 * (A,B) iff it holds an A before a B (A == B: at least two occurrences).  <= 32 pairs / 32 distinct activities. */
int siesta_index_build(siesta_log* log, const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs,
                       siesta_index** out);
/* After siesta_log_append: a new index on new_log (the log the append returned, or one grown from it by later appends)
 * that follows the appended events.  Neither call modifies `index`: it stays valid on its own log and keeps answering
 * siesta_intersect / siesta_candidates while the new one is built; the caller swaps handles as with the log.  `index`'s log
 * must still be alive during the call.  Both are exact because an append only adds events after a trace's existing ones:
 * a trace keeps every pair it held, so no trace leaves a list, and traces the batch did not list are unchanged.
 * SIESTA_E_INVALID (nothing allocated, *out untouched, `index` unchanged): a null argument, new_log on another context or
 * with fewer traces than the index's log, or the call-specific cases below.  *kernel_ms (may be NULL) = device time between
 * CUDA events on the context's stream after the host -> device copies (work other threads enqueue on the context during
 * the call is counted too).
 *
 * siesta_index_append: list p = index's list p UNION delta list p (ascending, duplicate-free).  Delta list p =
 * delta_trace_idx[delta_off[p] .. delta_off[p+1]), strictly ascending trace indices of new_log, in the index's pair order;
 * it may repeat traces the old list holds (index.parquet rows of a batch name traces that were listed before).
 * delta_trace_idx may be NULL when every delta list is empty.  The result counts as a loaded index, whatever `index` was.
 * Refused: delta_off[0] != 0, delta_off decreasing, a delta list not strictly ascending or holding an index outside
 * [0, new_log's n_traces). */
int siesta_index_append(siesta_index* index, siesta_log* new_log, const int64_t* delta_off, const int64_t* delta_trace_idx,
                        siesta_index** out, double* kernel_ms);
/* siesta_index_refresh: built indexes only (siesta_index_build or an earlier refresh).  Re-derives, under the SeqTable
 * view on new_log, the membership of the traces the batch listed (trace_idx[n_listed] exactly as passed to
 * siesta_log_append, strictly ascending; NULL when n_listed == 0) and merges it into the old lists: the result equals
 * siesta_index_build(new_log, same pairs) and is a built index.  One case re-flags EVERY trace: when the index's log held
 * activity ids outside its alphabet (not every id of the log lies in [0, n_activities)) and new_log's larger alphabet
 * covers an activity one of the pairs names, unlisted traces that hold such an id gain the pair, as
 * siesta_index_build counts them now; the call then costs a full build.  Refused: a loaded index (siesta_index_load or
 * siesta_index_append), n_listed < 0, trace_idx not strictly ascending or outside [0, new_log's n_traces), or not
 * listing every new trace [index's n_traces, new_log's n_traces).  SIESTA_E_UNSUPPORTED as siesta_index_build when the
 * pairs mention more than 32 activities of new_log's alphabet. */
int siesta_index_refresh(siesta_index* index, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed,
                         siesta_index** out, double* kernel_ms);
void siesta_index_free(siesta_index* index);
int64_t siesta_index_list_len(const siesta_index* index, int32_t pair);
int siesta_index_get_list(const siesta_index* index, int32_t pair, int64_t* out, int64_t cap);
/* Intersection of lists pair_ids[0..n): ascending trace indices, ready to be siesta_detect's `cand`. */
int siesta_intersect(siesta_index* index, const int32_t* pair_ids, int32_t n, int64_t* out, int64_t cap, int64_t* out_n);
/* Same, result left in HBM (*d_out, free with siesta_device_free) for siesta_detect_device's d_cand. */
int siesta_intersect_device(siesta_index* index, const int32_t* pair_ids, int32_t n, int64_t** d_out, int64_t* out_n,
                            double* kernel_ms);
/* The candidate traces of a pattern with OR-expansions: the union over the expansions of the intersection of each
 * expansion's true-pair lists (QueryPlanPatternDetection.getMiddleResults :146-164 merges the per-expansion results).
 * Expansion x uses lists pair_ids[exp_off[x] .. exp_off[x+1]).  Ascending trace indices. */
int siesta_candidates_device(siesta_index* index, const int32_t* exp_off, const int32_t* pair_ids, int32_t n_expansions,
                             int64_t** d_out, int64_t* out_n, double* kernel_ms);
int siesta_candidates(siesta_index* index, const int32_t* exp_off, const int32_t* pair_ids, int32_t n_expansions,
                      int64_t* out, int64_t cap, int64_t* out_n);
void siesta_device_free(siesta_log* log, void* d_ptr);

/* ------------------------------------------------------- declare counting */
/* Kernel K3.  Replaces the per-trace counting of the declare plans (declare/queryPlans/):
 *   existence/QueryPlanExistences.java  createMapForSingle :136-142, extractUniqueTracesSingle :150-158,
 *                                       joinUnionTraces :164-179 (over S3Connector.queryIndexTableDeclare :389-404)
 *   orderedRelations/QueryPlanOrderedRelations.java  joinTables :97-116, evaluateConstraint :127-151 with
 *                                       OrderedRelationsUtilityFunctions.countResponse / countPrecedence :25-44
 *   position/QueryPlanPositions.java    execute :51-79
 * over the SeqTable view of the pair index (a trace is listed under (A,B) iff it holds an A before a B).
 * The result is ONE packed int64 array so that the multi-GPU combine is a single sum all-reduce:
 *   tot[A] uniq[A] first[A] last[A] hist[A][k_cap+1] co[A][A] ordered[A][A] response[A][A] precedence[A][A]
 *   alt_response[A][A] alt_precedence[A][A] chain_response[A][A] chain_precedence[A][A]
 *   hist_overflow n_nonempty_traces
 * alt_* / chain_*: the alternate and chain modes (orderedRelations/QueryPlanOrderedRelationsAlternate.java,
 * ...Chain.java over OrderedRelationsUtilityFunctions.countResponseAlternate :51-60, countPrecedenceAlternate :67-76,
 * countResponseChain :83-89, countPrecedenceChain :96-102).
 * (meaning of each block: oracle/counting_oracle.cpp).  Supports and thresholds (one double division each:
 * QueryPlanExistences templates :188-438, QueryPlanOrderedRelations.filterBasedOnSupport :161-233) stay with
 * the caller.  n_activities <= 4096 (the result itself: eight A x A int64 matrices = 1 GB); alphabets above 104
 * activities use a kernel that works on the distinct activities of each trace, any trace length. */
int64_t siesta_declare_counts_size(int32_t n_activities, int32_t k_cap);
int siesta_declare_counts(siesta_log* log, int32_t k_cap, int64_t* out /* host, _size() values */, double* kernel_ms);
int siesta_declare_counts_device(siesta_log* log, int32_t k_cap, int64_t* d_out /* device */, void* stream,
                                 double* kernel_ms);
/* After siesta_log_append: the counts of new_log from those of old_log, recounting only the traces the batch listed.
 * Every block of the packed result is a sum of per-trace contributions and an append changes only the listed traces, so
 *     counts(new_log) = counts(old_log) - K3(old_log, listed old traces) + K3(new_log, listed traces)
 * in wrapping int64 arithmetic, with old_counts moved to new_log's alphabet (new rows and columns zero).  The result
 * equals siesta_declare_counts(new_log, k_cap) bit for bit.  Cost: 4 B per event of the listed traces in both logs,
 * 8 B per listed trace, one read and one write of the count array, 16 B per old trace for the check below.
 *   old_counts: siesta_declare_counts(old_log, k_cap) with the same k_cap, or an earlier refresh; laid out for old_log's
 *               alphabet (siesta_declare_counts_size(old A, k_cap) values).  out: laid out for new_log's alphabet.
 *   trace_idx:  exactly what siesta_log_append was given (strictly ascending, listing every new trace); across chained
 *               appends, the union of the batches' lists.  NULL when n_listed == 0.
 * old_log is only read and must stay alive during the call.  *kernel_ms (may be NULL) = device time between CUDA events on
 * the call's stream, from after the host -> device copy of trace_idx to the end of the merge (the check included).
 * One fallback: when old_log holds activity ids outside its alphabet (not every id lies in [0, n_activities)) and new_log's
 * alphabet is larger, unlisted traces may gain counted events, so the call counts new_log in full (still exact).
 * SIESTA_E_INVALID (nothing kept allocated, out untouched): a null argument, k_cap < 1, logs on different contexts, a
 * derived (siesta_log_filter_time / siesta_log_group) or block-cyclic log, new_log with fewer traces or a smaller alphabet
 * than old_log, trace_idx not strictly ascending inside [0, new_log's n_traces) or not listing every new trace, and an
 * unlisted trace whose length differs between the two logs (one device pass over both offset arrays).
 * SIESTA_E_UNSUPPORTED: new_log's alphabet above 4096, as siesta_declare_counts.
 * _device: d_old / d_out are device arrays; d_out may be d_old only when the alphabet did not grow.
 * Measured on one B200 at 1000 W (100 M traces x 50 events, 1 M touched traces x 5 events + 1 M new traces x 50 events):
 * 3.6 / 54 / 117 ms at 20 / 100 / 400 activities against 96 / 1 733 / 4 203 ms for siesta_declare_counts on the new log.
 * A batch that touches most traces is cheaper to count in full (both versions of every listed trace are counted). */
int siesta_declare_counts_refresh(siesta_log* old_log, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed,
                                  int32_t k_cap, const int64_t* old_counts /* host */, int64_t* out /* host */,
                                  double* kernel_ms);
int siesta_declare_counts_refresh_device(siesta_log* old_log, siesta_log* new_log, const int64_t* trace_idx, int64_t n_listed,
                                         int32_t k_cap, const int64_t* d_old, int64_t* d_out, void* stream, double* kernel_ms);

/* ------------------------------------------------------------- pair statistics */
/* Kernel K4.  The record /stats returns per consecutive pair of the pattern (QueryPlanStats.execute, model/Queries/
 * QueryPlans/QueryPlanStats.java:43-48; record: model/DBModel/Count.java:12-24).  In the reference the numbers are
 * READ from count.parquet, which the separate, un-vendored SIESTA preprocess writes; here they are computed from the
 * resident log under SIESTA's published pairing policy (non-overlapping skip-till-next-match pairs: first A, first B
 * after it, continue after that B).  PARITY UNPINNED: no source or golden vector of the preprocess is in the
 * reference repository (DESIGN.md).  Durations are ts_ms(B) - ts_ms(A); the sum of squares is exact (128 bit). */
typedef struct siesta_pair_count {
    int64_t count;
    int64_t sum_duration_ms;
    int64_t min_duration_ms; /* 0 when count == 0 */
    int64_t max_duration_ms;
    uint64_t sum_squares_lo, sum_squares_hi; /* sum of duration_ms^2 as a 128-bit integer */
} siesta_pair_count;
int siesta_pair_stats(siesta_log* log, const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs /* any number: passes of 32 */,
                      siesta_pair_count* out, double* kernel_ms);
/* Device form for the multi-GPU combine: d_out[8 * n_pairs] int64 = count, sum, min, max, and the sum of squares as
 * four 32-bit limbs (one per int64).  count / sum / limbs combine with a SUM all-reduce (carry-normalise afterwards),
 * min / max with MIN / MAX; with count == 0, min = INT64_MAX and max = INT64_MIN. */
int siesta_pair_stats_device(siesta_log* log, const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs,
                             int64_t* d_out, void* stream, double* kernel_ms);

/* ------------------------------------------------------------------- /explore */
/* Replaces QueryPlanExplorationAccurate.patternDetection (model/Queries/QueryPlans/Exploration/
 * QueryPlanExplorationAccurate.java:82-102) for every candidate continuation: the pattern (all "_" events, a
 * SimplePattern) extended by candidate c is detected with clearOccurrences(true) in every trace;
 * completions[c] = number of occurrences, sum_duration_ms[c] = sum over them of last.timestamp - first.timestamp in
 * milliseconds (Occurrence.getDuration, model/Occurrence.java:55-61, is this / 1000.0; the timestamps are those
 * siesta_detect reports: relative seconds * 1000 + the first filtered event on the EventTs route, the log's own
 * timestamps under SIESTA_F_EVT_POS).  The caller divides (average = sum / 1000.0 / completions) and sorts
 * (Proposition.compareTo, model/Proposition.java:51-60).  flags: 0 or SIESTA_F_EVT_POS.
 * One pass over the log serves all candidates (csrc/explore.cu); the result equals one siesta_detect with
 * SIESTA_F_RETURN_ALL per candidate. */
int siesta_explore_accurate(siesta_log* log, const int32_t* pattern_activities, int32_t n_pattern,
                            const int32_t* candidates, int32_t n_candidates, uint32_t flags,
                            int64_t* completions, int64_t* sum_duration_ms, double* kernel_ms);

/* ------------------------------------------------------------ why-not-match */
/* Replaces WhyNotMatchSASE.evaluate(SimplePattern, restEvents, uncertaintyPerEvent, step, k)
 * (model/WhyNotMatch/UsingSase/WhyNotMatchSASE.java:37-55; caller QueryPlanWhyNotMatch.execute :54-100, which
 * hands in the traces WITHOUT a true occurrence): for every candidate trace the events of the pattern's activities
 * are expanded into the uncertain stream (getUnCertainStream :63-83: every event at primary - u .. primary + u in
 * steps of `step`, clamped at 0, change = |shift|, stable sort by the shifted value; primary = epoch seconds, or the
 * position under SIESTA_F_EVT_POS: Event.getPrimaryMetric), the pattern's "normal" states run on it under
 * skip-till-any-match (S/engine/Engine.java:159-178, 341-350, 593-645) with the predicates of getNFA :91-152, and
 * the match of least total change is reported, the LAST such match in the engine's emission order (createResponse
 * :160-173: reduce keeps the later of two equal sums).  A trace without any match is not listed.
 *
 * The engine's behaviour is reproduced as it is, not as its comments describe it (oracle/wnm_oracle.cpp restates it
 * literally; DESIGN.md section 3, kernel W):
 *  - `change <= k - $2.change - ...` is only effective on the FIRST state: on every later state the predicate names
 *    its own state and PredicateOptimized.evaluate returns true for it (PredicateOptimized.java:348-350);
 *  - a constraint (posA, posB) with posA >= 1 is compared with the event that the runs of the same START took LAST at
 *    state posA, not with the run's own (Run.clone is shallow: the value vectors are shared by all runs that descend
 *    from one start, S/engine/Run.java:319-327, 332-355);
 *  - gap constraints count positions of the uncertain stream; `timestamp > $previous.timestamp` is only asked at a
 *    state a time constraint ends at.
 * Traces whose uncertain stream exceeds SIESTA_WNM_MAX_STREAM events are listed in unsupported_trace_idx, every
 * other trace is answered. */
#define SIESTA_WNM_GAP 0
#define SIESTA_WNM_TIME 1
#define SIESTA_WNM_WITHIN 0
#define SIESTA_WNM_ATLEAST 1
#define SIESTA_WNM_MAX_STREAM 1024
typedef struct siesta_wnm_constraint {
    int32_t pos_a, pos_b; /* Constraint.getPosA / getPosB, 0-based, pos_a < pos_b */
    int32_t kind;         /* SIESTA_WNM_GAP | SIESTA_WNM_TIME */
    int32_t method;       /* SIESTA_WNM_WITHIN | SIESTA_WNM_ATLEAST */
    int64_t value;        /* GapConstraint.getConstraint() / TimeConstraint.getConstraintInSeconds(), >= 0 */
} siesta_wnm_constraint;
typedef struct siesta_almost_matches {
    int64_t n_traces;        /* traces with an almost-match (AlmostMatch objects of the response) */
    int32_t n_states;        /* events per almost-match = length of the pattern */
    int64_t* trace_idx;      /* [n_traces] ascending (candidate order) */
    int32_t* total_change;   /* [n_traces] AlmostMatch.totalChange */
    int32_t* ev_pos;         /* [n_traces * n_states] index of the ORIGINAL event inside its trace */
    int32_t* ev_value;       /* [n_traces * n_states] UncertainTimeEvent.getTimestamp(): shifted primary metric */
    int32_t* ev_change;      /* [n_traces * n_states] UncertainTimeEvent.getChange() */
    int32_t* ev_stream_pos;  /* [n_traces * n_states] UncertainTimeEvent.getPosition(): index in the uncertain stream */
    int64_t n_unsupported;
    int64_t* unsupported_trace_idx;
    double kernel_ms;
} siesta_almost_matches;
int siesta_why_not_match(siesta_log* log, const int32_t* pattern_activities, int32_t n_pattern,
                         const siesta_wnm_constraint* constraints, int32_t n_constraints, int32_t uncertainty,
                         int32_t step, int32_t k, const int64_t* cand, int64_t n_cand, uint32_t flags,
                         siesta_almost_matches** out);
void siesta_almost_matches_free(siesta_almost_matches* m);

/* Number of kernels this library has launched in this process (bench.py's
 * gpu_launches). */
int64_t siesta_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* SIESTA_GPU_H */
