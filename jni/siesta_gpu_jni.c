/*
 * siesta_gpu_jni.c — the thin JNI layer between the reference's Java code and libsiesta_gpu (include/siesta_gpu.h).
 *
 * Native half of com.datalab.siesta.queryprocessor.SaseConnection.GpuNative (jni/java/...); GpuSaseConnector.java next
 * to it overrides the reference's verification seam
 *     List<Occurrences> SaseConnector.evaluate(SIESTAPattern, Map<String, List<Event>>, boolean onlyAppearances)
 * (SaseConnection/SaseConnector.java:48) on top of these calls.  Every failure of the library becomes a
 * java.lang.RuntimeException carrying siesta_last_error(), as the reference wraps the engine's exceptions
 * (SaseConnector.java:60-62).  Handles (contexts, logs, results) travel as jlong.
 *
 * Compiled in this repository against jni/stub/jni.h (no JDK in the image): a compile check of every call below.
 */
#include <jni.h>
#include <stdlib.h>
#include <string.h>

#include "../include/siesta_gpu.h"

#define NATIVE(ret, name) JNIEXPORT ret JNICALL Java_com_datalab_siesta_queryprocessor_SaseConnection_GpuNative_##name

static void throw_last(JNIEnv* env, const char* what) {
    char msg[768];
    const char* why = siesta_last_error();
    strncpy(msg, what, sizeof(msg) - 1);
    msg[sizeof(msg) - 1] = 0;
    strncat(msg, ": ", sizeof(msg) - strlen(msg) - 1);
    strncat(msg, why ? why : "", sizeof(msg) - strlen(msg) - 1);
    jclass rte = (*env)->FindClass(env, "java/lang/RuntimeException");
    if (rte) (*env)->ThrowNew(env, rte, msg);
}

static void throw_class(JNIEnv* env, const char* cls, const char* msg) {
    jclass c = (*env)->FindClass(env, cls);
    if (c) (*env)->ThrowNew(env, c, msg);
}

/* long init(int[] deviceIds): one process drives all GPUs (siesta_multi_init) */
NATIVE(jlong, init)(JNIEnv* env, jclass cls, jintArray deviceIds) {
    (void)cls;
    const jsize n = (*env)->GetArrayLength(env, deviceIds);
    jint* ids = (*env)->GetIntArrayElements(env, deviceIds, NULL);
    siesta_multi* m = NULL;
    const int rc = siesta_multi_init((const int32_t*)ids, (int32_t)n, &m);
    (*env)->ReleaseIntArrayElements(env, deviceIds, ids, JNI_ABORT);
    if (rc != SIESTA_OK) {
        throw_last(env, "siesta_multi_init");
        return 0;
    }
    return (jlong)(intptr_t)m;
}

NATIVE(void, shutdown)(JNIEnv* env, jclass cls, jlong multi) {
    (void)env; (void)cls;
    siesta_multi_shutdown((siesta_multi*)(intptr_t)multi);
}

/* int[] patternCompile(int[] symbols, long[] constraints, boolean onlyAppearances) -> the siesta_nfa as int words
 *   symbols:     3 ints per EventSymbol  (activity id, position, symbol code SIESTA_SYM_*)
 *   constraints: 6 longs per Constraint  (posA, posB, kind, method, value, granularity)
 * = ComplexPattern.getNfa / getNfaWithoutConstraints (ComplexPattern.java:194-283) */
NATIVE(jintArray, patternCompile)(JNIEnv* env, jclass cls, jintArray symbols, jlongArray constraints, jboolean onlyAppearances) {
    (void)cls;
    const jsize ns = (*env)->GetArrayLength(env, symbols) / 3, nc = (*env)->GetArrayLength(env, constraints) / 6;
    jint* s = (*env)->GetIntArrayElements(env, symbols, NULL);
    jlong* c = (*env)->GetLongArrayElements(env, constraints, NULL);
    siesta_event_symbol* es = (siesta_event_symbol*)calloc((size_t)(ns ? ns : 1), sizeof(*es));
    siesta_constraint* cs = (siesta_constraint*)calloc((size_t)(nc ? nc : 1), sizeof(*cs));
    for (jsize i = 0; i < ns; ++i) {
        es[i].activity = s[3 * i];
        es[i].position = s[3 * i + 1];
        es[i].symbol = s[3 * i + 2];
    }
    for (jsize i = 0; i < nc; ++i) {
        cs[i].pos_a = (int32_t)c[6 * i];
        cs[i].pos_b = (int32_t)c[6 * i + 1];
        cs[i].kind = (int32_t)c[6 * i + 2];
        cs[i].method = (int32_t)c[6 * i + 3];
        cs[i].value = c[6 * i + 4];
        cs[i].granularity = (int32_t)c[6 * i + 5];
    }
    siesta_nfa nfa;
    memset(&nfa, 0, sizeof(nfa));
    const int rc = siesta_pattern_compile(es, (int32_t)ns, cs, (int32_t)nc, onlyAppearances ? 1 : 0, &nfa);
    free(es);
    free(cs);
    (*env)->ReleaseIntArrayElements(env, symbols, s, JNI_ABORT);
    (*env)->ReleaseLongArrayElements(env, constraints, c, JNI_ABORT);
    if (rc != SIESTA_OK) {
        throw_last(env, "siesta_pattern_compile");
        return NULL;
    }
    const jsize words = (jsize)(sizeof(nfa) / sizeof(jint));
    jintArray out = (*env)->NewIntArray(env, words);
    if (out) (*env)->SetIntArrayRegion(env, out, 0, words, (const jint*)&nfa);
    return out;
}

static int nfa_from(JNIEnv* env, jintArray words, siesta_nfa* nfa) {
    if ((size_t)(*env)->GetArrayLength(env, words) * sizeof(jint) != sizeof(*nfa)) return 0;
    jint* w = (*env)->GetIntArrayElements(env, words, NULL);
    memcpy(nfa, w, sizeof(*nfa));
    (*env)->ReleaseIntArrayElements(env, words, w, JNI_ABORT);
    return 1;
}

/* long logLoad(long multi, long[] traceOff, int[] act, long[] tsMs, int nActivities): resident, sharded CSR log */
NATIVE(jlong, logLoad)(JNIEnv* env, jclass cls, jlong multi, jlongArray traceOff, jintArray act, jlongArray tsMs, jint nActivities) {
    (void)cls;
    const jsize nt = (*env)->GetArrayLength(env, traceOff) - 1, ne = (*env)->GetArrayLength(env, act);
    /* critical sections: the arrays are only read, by a plain memcpy to the devices */
    jlong* off = (jlong*)(*env)->GetPrimitiveArrayCritical(env, traceOff, NULL);
    jint* a = (jint*)(*env)->GetPrimitiveArrayCritical(env, act, NULL);
    jlong* ts = (jlong*)(*env)->GetPrimitiveArrayCritical(env, tsMs, NULL);
    siesta_multi_log* log = NULL;
    const int rc = siesta_multi_log_load((siesta_multi*)(intptr_t)multi, (const int64_t*)off, (const int32_t*)a, (const int64_t*)ts,
                                         (int64_t)nt, (int64_t)ne, (int32_t)nActivities, &log);
    (*env)->ReleasePrimitiveArrayCritical(env, tsMs, ts, JNI_ABORT);
    (*env)->ReleasePrimitiveArrayCritical(env, act, a, JNI_ABORT);
    (*env)->ReleasePrimitiveArrayCritical(env, traceOff, off, JNI_ABORT);
    if (rc != SIESTA_OK) {
        throw_last(env, "siesta_multi_log_load");
        return 0;
    }
    return (jlong)(intptr_t)log;
}

/* long logAppend(long log, long[] traceIdx, long[] batchOff, int[] act, long[] tsMs, long nNewTraces, int nActivities):
 * a new resident log with the batch appended (siesta_multi_log_append); the old handle stays valid until logFree.
 * The arrays are copied out first (Get<Type>ArrayRegion), so none is pinned while the devices rebuild their shards. */
NATIVE(jlong, logAppend)(JNIEnv* env, jclass cls, jlong log, jlongArray traceIdx, jlongArray batchOff, jintArray act, jlongArray tsMs,
                         jlong nNewTraces, jint nActivities) {
    (void)cls;
    const jsize nl = (*env)->GetArrayLength(env, traceIdx), ne = (*env)->GetArrayLength(env, act);
    int64_t* off = NULL;
    if ((*env)->GetArrayLength(env, batchOff) == nl + 1) {
        off = (int64_t*)malloc(sizeof(int64_t) * (size_t)(nl + 1));
        if (!off) {
            throw_class(env, "java/lang/OutOfMemoryError", "logAppend: host copy of the batch");
            return 0;
        }
        (*env)->GetLongArrayRegion(env, batchOff, 0, nl + 1, (jlong*)off);
    }
    /* the library copies batchOff[nl] events: it must be exactly the arrays' length */
    if (!off || (*env)->GetArrayLength(env, tsMs) != ne || off[nl] != (int64_t)ne) {
        free(off);
        throw_class(env, "java/lang/IllegalArgumentException",
                    "logAppend: batchOff needs traceIdx.length + 1 entries ending at act.length, tsMs act.length entries");
        return 0;
    }
    int64_t* idx = (int64_t*)malloc(sizeof(int64_t) * (size_t)(nl ? nl : 1));
    int32_t* a = (int32_t*)malloc(sizeof(int32_t) * (size_t)(ne ? ne : 1));
    int64_t* ts = (int64_t*)malloc(sizeof(int64_t) * (size_t)(ne ? ne : 1));
    if (!idx || !a || !ts) {
        free(off); free(idx); free(a); free(ts);
        throw_class(env, "java/lang/OutOfMemoryError", "logAppend: host copy of the batch");
        return 0;
    }
    (*env)->GetLongArrayRegion(env, traceIdx, 0, nl, (jlong*)idx);
    (*env)->GetIntArrayRegion(env, act, 0, ne, (jint*)a);
    (*env)->GetLongArrayRegion(env, tsMs, 0, ne, (jlong*)ts);
    siesta_multi_log* out = NULL;
    const int rc = siesta_multi_log_append((siesta_multi_log*)(intptr_t)log, idx, off, (int64_t)nl, a, ts, (int64_t)nNewTraces,
                                           (int32_t)nActivities, &out);
    free(off); free(idx); free(a); free(ts);
    if (rc != SIESTA_OK) {
        throw_last(env, "siesta_multi_log_append");
        return 0;
    }
    return (jlong)(intptr_t)out;
}

NATIVE(void, logFree)(JNIEnv* env, jclass cls, jlong log) {
    (void)env; (void)cls;
    siesta_multi_log_free((siesta_multi_log*)(intptr_t)log);
}

/* long detect(long log, int[] nfa, int flags) -> handle of a siesta_matches (free with matchesFree)
 * = SaseConnector.evaluate + occurrences.forEach(clearOccurrences(returnAll)) over all traces of the log */
NATIVE(jlong, detect)(JNIEnv* env, jclass cls, jlong log, jintArray nfaWords, jint flags) {
    (void)cls;
    siesta_nfa nfa;
    if (!nfa_from(env, nfaWords, &nfa)) {
        jclass iae = (*env)->FindClass(env, "java/lang/IllegalArgumentException");
        if (iae) (*env)->ThrowNew(env, iae, "nfa: not the words patternCompile returned");
        return 0;
    }
    siesta_matches* m = NULL;
    if (siesta_multi_detect((siesta_multi_log*)(intptr_t)log, &nfa, (uint32_t)flags, &m) != SIESTA_OK) {
        throw_last(env, "siesta_multi_detect");
        return 0;
    }
    return (jlong)(intptr_t)m;
}

/* long evaluateEvents(long multi, long[] traceOff, int[] act, long[] tsMs, int nActivities, int[] nfa, int flags):
 * the literal seam - the events of THIS request arrive from the Java heap (SaseConnector.java:48-51) */
NATIVE(jlong, evaluateEvents)(JNIEnv* env, jclass cls, jlong multi, jlongArray traceOff, jintArray act, jlongArray tsMs,
                              jint nActivities, jintArray nfaWords, jint flags) {
    const jlong log = Java_com_datalab_siesta_queryprocessor_SaseConnection_GpuNative_logLoad(env, cls, multi, traceOff, act, tsMs, nActivities);
    if (!log || (*env)->ExceptionCheck(env)) return 0;
    const jlong m = Java_com_datalab_siesta_queryprocessor_SaseConnection_GpuNative_detect(env, cls, log, nfaWords, flags);
    siesta_multi_log_free((siesta_multi_log*)(intptr_t)log);
    return m;
}

/* long[] matchesSizes(long m) -> { n_traces, n_occurrences, n_events, n_matches_emitted, n_ref_errors, n_unsupported } */
NATIVE(jlongArray, matchesSizes)(JNIEnv* env, jclass cls, jlong mh) {
    (void)cls;
    const siesta_matches* m = (const siesta_matches*)(intptr_t)mh;
    const jlong v[6] = {m->n_traces, m->n_occurrences, m->n_events, m->n_matches_emitted, m->n_ref_errors, m->n_unsupported};
    jlongArray out = (*env)->NewLongArray(env, 6);
    if (out) (*env)->SetLongArrayRegion(env, out, 0, 6, v);
    return out;
}

/* long[] matchesLongs(long m, int which): 0 trace_idx, 1 occ_off, 2 ev_off, 3 ev_ts_ms, 4 err_trace_idx,
 * 5 unsupported_trace_idx (traces beyond the GPU engine's limits: evaluate them with the reference's engine) */
NATIVE(jlongArray, matchesLongs)(JNIEnv* env, jclass cls, jlong mh, jint which) {
    (void)cls;
    const siesta_matches* m = (const siesta_matches*)(intptr_t)mh;
    const int64_t* src = NULL;
    int64_t n = 0;
    switch (which) {
        case 0: src = m->trace_idx; n = m->n_traces; break;
        case 1: src = m->occ_off; n = m->n_traces + 1; break;
        case 2: src = m->ev_off; n = m->n_occurrences + 1; break;
        case 3: src = m->ev_ts_ms; n = src ? m->n_events : 0; break;
        case 4: src = m->err_trace_idx; n = m->n_ref_errors; break;
        case 5: src = m->unsupported_trace_idx; n = m->n_unsupported; break;
        default: break;
    }
    if (n > 0x7fffffff) {   /* a Java array holds < 2^31 elements: ask for a narrower candidate list */
        jclass rte = (*env)->FindClass(env, "java/lang/RuntimeException");
        if (rte) (*env)->ThrowNew(env, rte, "result column longer than a Java array");
        return NULL;
    }
    jlongArray out = (*env)->NewLongArray(env, (jsize)n);
    if (out && n) (*env)->SetLongArrayRegion(env, out, 0, (jsize)n, (const jlong*)src);
    return out;
}

/* int[] matchesInts(long m, int which): 0 ev_pos, 1 ev_rank, 2 ev_act */
NATIVE(jintArray, matchesInts)(JNIEnv* env, jclass cls, jlong mh, jint which) {
    (void)cls;
    const siesta_matches* m = (const siesta_matches*)(intptr_t)mh;
    const int32_t* src = which == 0 ? m->ev_pos : (which == 1 ? m->ev_rank : (which == 2 ? m->ev_act : NULL));
    const int64_t n = src ? m->n_events : 0;
    if (n > 0x7fffffff) {
        jclass rte = (*env)->FindClass(env, "java/lang/RuntimeException");
        if (rte) (*env)->ThrowNew(env, rte, "result column longer than a Java array");
        return NULL;
    }
    jintArray out = (*env)->NewIntArray(env, (jsize)n);
    if (out && n) (*env)->SetIntArrayRegion(env, out, 0, (jsize)n, (const jint*)src);
    return out;
}

NATIVE(void, matchesFree)(JNIEnv* env, jclass cls, jlong mh) {
    (void)env; (void)cls;
    siesta_matches_free((siesta_matches*)(intptr_t)mh);
}

/* long[] declareCounts(long log, int kCap): the packed integer matrices behind /declare (layout: siesta_gpu.h) */
NATIVE(jlongArray, declareCounts)(JNIEnv* env, jclass cls, jlong log, jint nActivities, jint kCap) {
    (void)cls;
    const int64_t n = siesta_declare_counts_size((int32_t)nActivities, (int32_t)kCap);
    int64_t* buf = (int64_t*)malloc((size_t)(n > 0 ? n : 1) * sizeof(int64_t));
    double ms = 0;
    const int rc = buf ? siesta_multi_declare_counts((siesta_multi_log*)(intptr_t)log, (int32_t)kCap, buf, &ms) : SIESTA_E_NOMEM;
    jlongArray out = NULL;
    if (rc != SIESTA_OK) throw_last(env, "siesta_multi_declare_counts");
    else {
        out = (*env)->NewLongArray(env, (jsize)n);
        if (out) (*env)->SetLongArrayRegion(env, out, 0, (jsize)n, (const jlong*)buf);
    }
    free(buf);
    return out;
}

/* long whyNotMatch(long log, int[] pattern, long[] constraints, int uncertainty, int step, int k, long[] cand, int flags):
 * WhyNotMatchSASE.evaluate (model/WhyNotMatch/UsingSase/WhyNotMatchSASE.java:37-55) over the candidate traces of a
 * resident log.  constraints: 5 longs per Constraint (posA, posB, kind SIESTA_WNM_GAP|TIME, method SIESTA_WNM_WITHIN|ATLEAST,
 * value: positions, or TimeConstraint.getConstraintInSeconds()); cand: ascending trace indices, null = every trace. */
NATIVE(jlong, whyNotMatch)(JNIEnv* env, jclass cls, jlong log, jintArray pattern, jlongArray constraints, jint uncertainty, jint step,
                           jint k, jlongArray cand, jint flags) {
    (void)cls;
    const jsize m = (*env)->GetArrayLength(env, pattern), nc = (*env)->GetArrayLength(env, constraints) / 5;
    const jsize ncand = cand ? (*env)->GetArrayLength(env, cand) : 0;
    jint* p = (*env)->GetIntArrayElements(env, pattern, NULL);
    jlong* c = (*env)->GetLongArrayElements(env, constraints, NULL);
    jlong* cd = cand ? (*env)->GetLongArrayElements(env, cand, NULL) : NULL;
    siesta_wnm_constraint* cons = (siesta_wnm_constraint*)malloc(sizeof(siesta_wnm_constraint) * (size_t)(nc > 0 ? nc : 1));
    siesta_almost_matches* out = NULL;
    int rc = SIESTA_E_NOMEM;
    if (cons) {
        for (jsize i = 0; i < nc; ++i) {
            cons[i].pos_a = (int32_t)c[5 * i];
            cons[i].pos_b = (int32_t)c[5 * i + 1];
            cons[i].kind = (int32_t)c[5 * i + 2];
            cons[i].method = (int32_t)c[5 * i + 3];
            cons[i].value = (int64_t)c[5 * i + 4];
        }
        static const int64_t none = 0;   /* an empty candidate list is "no trace", not "every trace" */
        rc = siesta_multi_why_not_match((siesta_multi_log*)(intptr_t)log, (const int32_t*)p, (int32_t)m, cons, (int32_t)nc, (int32_t)uncertainty,
                                        (int32_t)step, (int32_t)k, cand ? (ncand ? (const int64_t*)cd : &none) : NULL, (int64_t)ncand,
                                        (uint32_t)flags, &out);
    }
    free(cons);
    (*env)->ReleaseIntArrayElements(env, pattern, p, JNI_ABORT);
    (*env)->ReleaseLongArrayElements(env, constraints, c, JNI_ABORT);
    if (cd) (*env)->ReleaseLongArrayElements(env, cand, cd, JNI_ABORT);
    if (rc != SIESTA_OK) {
        throw_last(env, "siesta_multi_why_not_match");
        return 0;
    }
    return (jlong)(intptr_t)out;
}

/* long[] almostLongs(long a, int which): 0 trace_idx, 1 unsupported_trace_idx */
NATIVE(jlongArray, almostLongs)(JNIEnv* env, jclass cls, jlong ah, jint which) {
    (void)cls;
    const siesta_almost_matches* a = (const siesta_almost_matches*)(intptr_t)ah;
    const int64_t* src = which == 0 ? a->trace_idx : a->unsupported_trace_idx;
    const int64_t n = which == 0 ? a->n_traces : a->n_unsupported;
    jlongArray out = (*env)->NewLongArray(env, (jsize)n);
    if (out && n) (*env)->SetLongArrayRegion(env, out, 0, (jsize)n, (const jlong*)src);
    return out;
}

/* int[] almostInts(long a, int which): 0 total_change [n], then n * n_states each: 1 ev_pos, 2 ev_value, 3 ev_change, 4 ev_stream_pos */
NATIVE(jintArray, almostInts)(JNIEnv* env, jclass cls, jlong ah, jint which) {
    (void)cls;
    const siesta_almost_matches* a = (const siesta_almost_matches*)(intptr_t)ah;
    const int32_t* src = which == 0 ? a->total_change : which == 1 ? a->ev_pos : which == 2 ? a->ev_value : which == 3 ? a->ev_change : a->ev_stream_pos;
    const int64_t n = which == 0 ? a->n_traces : a->n_traces * a->n_states;
    if (n > 0x7fffffff) {
        jclass rte = (*env)->FindClass(env, "java/lang/RuntimeException");
        if (rte) (*env)->ThrowNew(env, rte, "result column longer than a Java array");
        return NULL;
    }
    jintArray out = (*env)->NewIntArray(env, (jsize)n);
    if (out && n) (*env)->SetIntArrayRegion(env, out, 0, (jsize)n, (const jint*)src);
    return out;
}

NATIVE(void, almostFree)(JNIEnv* env, jclass cls, jlong ah) {
    (void)env; (void)cls;
    siesta_almost_matches_free((siesta_almost_matches*)(intptr_t)ah);
}
