"""Loads libsiesta_gpu.so (built in-tree by csrc/Makefile) and declares the C-ABI of include/siesta_gpu.h.

There is no CPU fallback: a missing library or a missing sm_100 device raises."""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SIESTA_GPU_LIB") or os.path.join(_HERE, "libsiesta_gpu.so")  # override: instrumented builds
_lib = None

EXPORTS = [
    "siesta_last_error", "siesta_pattern_compile", "siesta_init", "siesta_shutdown", "siesta_log_load",
    "siesta_log_wrap_device", "siesta_log_free", "siesta_log_n_traces", "siesta_log_n_events", "siesta_detect",
    "siesta_matches_free", "siesta_evaluate_events", "siesta_evaluate_events_act8", "siesta_detect_device", "siesta_detect_device_begin", "siesta_detect_device_finish", "siesta_dev_matches_free",
    "siesta_kernel_launches", "siesta_declare_counts_size", "siesta_declare_counts", "siesta_declare_counts_device",
    "siesta_index_load", "siesta_index_build", "siesta_index_free", "siesta_index_list_len", "siesta_index_get_list",
    "siesta_intersect", "siesta_intersect_device", "siesta_device_free", "siesta_pattern_extract_pairs",
    "siesta_candidates", "siesta_candidates_device", "siesta_pair_stats", "siesta_pair_stats_device",
    "siesta_explore_accurate", "siesta_why_not_match", "siesta_almost_matches_free", "siesta_log_set_first_trace", "siesta_log_set_blocks",
    "siesta_exchange_create", "siesta_exchange_export", "siesta_exchange_import", "siesta_exchange_connect_local",
    "siesta_exchange_free", "siesta_exchange_required_bytes", "siesta_detect_allgather", "siesta_exchange_allreduce_i64",
    "siesta_multi_init", "siesta_multi_shutdown", "siesta_multi_n_devices", "siesta_multi_log_load", "siesta_multi_log_free",
    "siesta_multi_log_shard", "siesta_multi_detect", "siesta_multi_declare_counts", "siesta_multi_why_not_match",
    "siesta_log_filter_time", "siesta_log_group", "siesta_log_source_events",
    "siesta_log_append", "siesta_log_read", "siesta_multi_log_append", "siesta_index_append", "siesta_index_refresh",
]


class SiestaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libsiesta_gpu error {code}: {msg}")
        self.code = code


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
                          "(python __graft_entry__.py build). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    i32, i64, u32, vp = C.c_int32, C.c_int64, C.c_uint32, C.c_void_p
    P = C.POINTER
    L.siesta_last_error.restype = C.c_char_p
    L.siesta_pattern_compile.argtypes = [P(_abi.EventSymbolC), i32, P(_abi.ConstraintC), i32, i32, P(_abi.Nfa)]
    L.siesta_init.argtypes = [i32, P(vp)]
    L.siesta_shutdown.argtypes = [vp]
    L.siesta_shutdown.restype = None
    L.siesta_log_load.argtypes = [vp, vp, vp, vp, i64, i64, i32, P(vp)]
    L.siesta_log_wrap_device.argtypes = [vp, vp, vp, vp, i64, i64, i32, i32, P(vp)]
    L.siesta_log_set_first_trace.argtypes = [vp, i64]
    L.siesta_log_set_first_trace.restype = None
    L.siesta_log_set_blocks.argtypes = [vp, i32, P(i64), P(i64)]
    L.siesta_log_free.argtypes = [vp]
    L.siesta_log_free.restype = None
    L.siesta_log_n_traces.argtypes = [vp]
    L.siesta_log_n_traces.restype = i64
    L.siesta_log_n_events.argtypes = [vp]
    L.siesta_log_n_events.restype = i64
    L.siesta_detect.argtypes = [vp, P(_abi.Nfa), vp, i64, u32, P(P(_abi.Matches))]
    L.siesta_matches_free.argtypes = [P(_abi.Matches)]
    L.siesta_matches_free.restype = None
    L.siesta_evaluate_events.argtypes = [vp, vp, vp, vp, i64, i64, i32, P(_abi.Nfa), u32, P(P(_abi.Matches))]
    L.siesta_evaluate_events_act8.argtypes = [vp, vp, vp, vp, i64, i64, i32, P(_abi.Nfa), u32, P(P(_abi.Matches))]
    L.siesta_detect_device.argtypes = [vp, P(_abi.Nfa), vp, i64, u32, vp, P(_abi.DevMatches)]
    L.siesta_detect_device_begin.argtypes = [vp, P(_abi.Nfa), vp, i64, u32, vp, P(vp)]
    L.siesta_detect_device_finish.argtypes = [vp, P(_abi.DevMatches)]
    L.siesta_dev_matches_free.argtypes = [P(_abi.DevMatches)]
    L.siesta_dev_matches_free.restype = None
    L.siesta_kernel_launches.restype = i64
    L.siesta_declare_counts_size.argtypes = [i32, i32]
    L.siesta_declare_counts_size.restype = i64
    L.siesta_declare_counts.argtypes = [vp, i32, vp, P(C.c_double)]
    L.siesta_declare_counts_device.argtypes = [vp, i32, vp, vp, P(C.c_double)]
    L.siesta_index_load.argtypes = [vp, i32, vp, vp, vp, vp, P(vp)]
    L.siesta_index_build.argtypes = [vp, vp, vp, i32, P(vp)]
    L.siesta_index_append.argtypes = [vp, vp, vp, vp, P(vp), P(C.c_double)]
    L.siesta_index_refresh.argtypes = [vp, vp, vp, i64, P(vp), P(C.c_double)]
    L.siesta_index_free.argtypes = [vp]
    L.siesta_index_free.restype = None
    L.siesta_index_list_len.argtypes = [vp, i32]
    L.siesta_index_list_len.restype = i64
    L.siesta_index_get_list.argtypes = [vp, i32, vp, i64]
    L.siesta_intersect.argtypes = [vp, vp, i32, vp, i64, P(i64)]
    L.siesta_intersect_device.argtypes = [vp, vp, i32, P(vp), P(i64), P(C.c_double)]
    P32 = P(i32)
    L.siesta_pattern_extract_pairs.argtypes = [P(_abi.EventSymbolC), i32, P(_abi.ConstraintC), i32, i32, i32, i32, P32,
                                               P32, P32, P32, P32, P32, P32]
    L.siesta_candidates.argtypes = [vp, vp, vp, i32, vp, i64, P(i64)]
    L.siesta_candidates_device.argtypes = [vp, vp, vp, i32, P(vp), P(i64), P(C.c_double)]
    L.siesta_pair_stats.argtypes = [vp, vp, vp, i32, P(_abi.PairCount), P(C.c_double)]
    L.siesta_pair_stats_device.argtypes = [vp, vp, vp, i32, vp, vp, P(C.c_double)]
    L.siesta_explore_accurate.argtypes = [vp, vp, i32, vp, i32, u32, vp, vp, P(C.c_double)]
    L.siesta_why_not_match.argtypes = [vp, vp, i32, vp, i32, i32, i32, i32, vp, i64, u32, P(P(_abi.AlmostMatches))]
    L.siesta_multi_why_not_match.argtypes = [vp, vp, i32, vp, i32, i32, i32, i32, vp, i64, u32, P(P(_abi.AlmostMatches))]
    L.siesta_almost_matches_free.argtypes = [P(_abi.AlmostMatches)]
    L.siesta_almost_matches_free.restype = None
    L.siesta_exchange_create.argtypes = [vp, i32, i32, i64, P(vp)]
    L.siesta_exchange_export.argtypes = [vp, vp]
    L.siesta_exchange_import.argtypes = [vp, i32, vp]
    L.siesta_exchange_connect_local.argtypes = [vp, i32, vp]
    L.siesta_exchange_free.argtypes = [vp]
    L.siesta_exchange_free.restype = None
    L.siesta_exchange_required_bytes.argtypes = [vp, P(_abi.Nfa), u32]
    L.siesta_exchange_required_bytes.restype = i64
    L.siesta_detect_allgather.argtypes = [vp, P(_abi.Nfa), u32, vp, P(_abi.DevMatches), P(_abi.ExchangeStats)]
    L.siesta_exchange_allreduce_i64.argtypes = [vp, vp, i64, i32, vp]
    L.siesta_multi_init.argtypes = [vp, i32, P(vp)]
    L.siesta_multi_shutdown.argtypes = [vp]
    L.siesta_multi_shutdown.restype = None
    L.siesta_multi_n_devices.argtypes = [vp]
    L.siesta_multi_log_load.argtypes = [vp, vp, vp, vp, i64, i64, i32, P(vp)]
    L.siesta_multi_log_free.argtypes = [vp]
    L.siesta_multi_log_free.restype = None
    L.siesta_multi_log_shard.argtypes = [vp, i32]
    L.siesta_multi_log_shard.restype = vp
    L.siesta_multi_detect.argtypes = [vp, P(_abi.Nfa), u32, P(P(_abi.Matches))]
    L.siesta_multi_declare_counts.argtypes = [vp, i32, vp, P(C.c_double)]
    L.siesta_log_filter_time.argtypes = [vp, i64, i32, i64, i32, P(vp)]
    L.siesta_log_group.argtypes = [vp, vp, vp, i32, vp, i32, P(vp), vp, P(i32)]
    L.siesta_log_source_events.argtypes = [vp, vp]
    L.siesta_log_append.argtypes = [vp, vp, vp, i64, vp, vp, i64, i32, P(vp), P(C.c_double)]
    L.siesta_log_read.argtypes = [vp, i64, i64, vp, vp, vp]
    L.siesta_multi_log_append.argtypes = [vp, vp, vp, i64, vp, vp, i64, i32, P(vp)]
    L.siesta_device_free.argtypes = [vp, vp]
    L.siesta_device_free.restype = None
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise SiestaError(rc, lib().siesta_last_error().decode("utf-8", "replace"))
