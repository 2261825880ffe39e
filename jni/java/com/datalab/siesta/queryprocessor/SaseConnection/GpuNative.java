package com.datalab.siesta.queryprocessor.SaseConnection;

/**
 * Java half of jni/siesta_gpu_jni.c: the native methods of libsiesta_gpu (include/siesta_gpu.h).
 * Handles are jlong; every failure of the library arrives as a RuntimeException (as SaseConnector wraps the engine's
 * exceptions, SaseConnector.java:60-62).  NOT compiled in the repository this file ships in (no JDK in its image).
 */
final class GpuNative {
    static { System.loadLibrary("siesta_gpu_jni"); }

    // flags of include/siesta_gpu.h
    static final int F_RETURN_ALL = 1, F_ONLY_APPEARANCES = 2, F_EVT_POS = 8, F_NO_EVENT_COLUMNS = 16, F_COUNT_MATCHES = 32;
    // symbol / constraint codes of include/siesta_gpu.h
    static final int SYM_NORMAL = 0, SYM_PLUS = 1, SYM_STAR = 2, SYM_NOT = 3, SYM_OR = 4;
    static final int CONSTRAINT_GAP = 0, CONSTRAINT_TIME = 1, METHOD_WITHIN = 0, METHOD_ATLEAST = 1;
    static final int GRAN_SECONDS = 0, GRAN_MINUTES = 1, GRAN_HOURS = 2;

    static native long init(int[] deviceIds);
    static native void shutdown(long multi);
    static native int[] patternCompile(int[] symbols, long[] constraints, boolean onlyAppearances);
    static native long logLoad(long multi, long[] traceOff, int[] act, long[] tsMs, int nActivities);
    static native void logFree(long log);
    // a new resident log = `log` + a batch (events of traceIdx[i] = act / tsMs[batchOff[i] .. batchOff[i + 1]), global
    // indices, >= the log's trace count for new traces); `log` stays valid until logFree
    static native long logAppend(long log, long[] traceIdx, long[] batchOff, int[] act, long[] tsMs, long nNewTraces, int nActivities);
    static native long detect(long log, int[] nfa, int flags);
    static native long evaluateEvents(long multi, long[] traceOff, int[] act, long[] tsMs, int nActivities, int[] nfa, int flags);
    static native long[] matchesSizes(long matches);
    static native long[] matchesLongs(long matches, int which);   // 0 trace_idx, 1 occ_off, 2 ev_off, 3 ev_ts_ms, 4 err_trace_idx, 5 unsupported_trace_idx
    static native int[] matchesInts(long matches, int which);     // 0 ev_pos, 1 ev_rank, 2 ev_act
    static native void matchesFree(long matches);
    static native long[] declareCounts(long log, int nActivities, int kCap);
    // the counts of newLog (grown from oldLog by logAppend) from oldLog's, recounting only the traces traceIdx lists
    // (global, ascending; the union over chained appends); oldCounts holds the counts of oldNActivities activities
    static native long[] declareCountsRefresh(long oldLog, long newLog, long[] traceIdx, long[] oldCounts, int oldNActivities,
                                              int nActivities, int kCap);
    // why-not-match (WhyNotMatchSASE.evaluate): constraints = 5 longs each (posA, posB, kind 0 gap | 1 time, method 0 within | 1 atleast, value)
    static native long whyNotMatch(long log, int[] pattern, long[] constraints, int uncertainty, int step, int k, long[] cand, int flags);
    static native long[] almostLongs(long almost, int which);    // 0 trace_idx, 1 unsupported_trace_idx
    static native int[] almostInts(long almost, int which);      // 0 total_change, 1 ev_pos, 2 ev_value, 3 ev_change, 4 ev_stream_pos
    static native void almostFree(long almost);

    private GpuNative() { }
}
