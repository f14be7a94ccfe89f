"""ctypes binding of libsearcharray_b200.so (the C ABI in include/searcharray_b200.h).

There is deliberately NO CPU fallback: if the CUDA library is missing or a call fails,
this raises.  (The shared library is built in-tree by searcharray_b200/build.py.)
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsearcharray_b200.so")

NO_TERM = 0xFFFFFFFF
NO_DOC = 0xFFFFFFFF
ALL_BITS = 0xFFFFFFFFFFFFFFFF

c_u64, c_u32, c_f32, c_int = ctypes.c_uint64, ctypes.c_uint32, ctypes.c_float, ctypes.c_int
P_u64, P_u32, P_f32 = ctypes.POINTER(c_u64), ctypes.POINTER(c_u32), ctypes.POINTER(c_f32)
P_void = ctypes.c_void_p


class SaStats(ctypes.Structure):
    _fields_ = [("term_kernel_ms", ctypes.c_double), ("term_kernel_launches", c_u64),
                ("term_kernel_queries", c_u64), ("topk_kernel_ms", ctypes.c_double),
                ("topk_kernel_launches", c_u64), ("phrase_kernel_ms", ctypes.c_double),
                ("phrase_kernel_launches", c_u64), ("total_launches", c_u64),
                ("phrase_cont_words", c_u64), ("phrase_matched_docs", c_u64)]


# name -> (restype, argtypes); must list EVERY symbol include/searcharray_b200.h declares
SIGNATURES = {
    "sa_last_error": (ctypes.c_char_p, []),
    "sa_device_count": (c_int, [ctypes.POINTER(c_int)]),
    "sa_host_alloc": (c_int, [ctypes.POINTER(P_void), c_u64]),
    "sa_host_free": (c_int, [P_void]),
    "sa_index_create": (c_int, [P_u64, c_u64, P_u64, P_u64, c_u32, P_f32, c_u64, c_u64, c_int,
                                ctypes.POINTER(P_void)]),
    "sa_index_destroy": (c_int, [P_void]),
    "sa_index_upload_mode": (c_int, [P_void, ctypes.POINTER(c_int)]),
    "sa_index_info": (c_int, [P_void, P_u64, P_u64, P_u32, P_u64]),
    "sa_docfreq": (c_int, [P_void, c_u32, P_u64]),
    "sa_index_set_rows": (c_int, [P_void, P_u64, c_u64]),
    "sa_docfreq_rows": (c_int, [P_void, c_u32, P_u64]),
    "sa_termfreqs": (c_int, [P_void, c_u32, c_u64, c_u64, P_f32]),
    "sa_score_term": (c_int, [P_void, c_u32, c_f32, c_f32, c_f32, c_f32, c_u64, c_u64, P_f32]),
    "sa_phrase_freqs": (c_int, [P_void, P_u32, c_u32, c_u32, c_u64, c_u64, P_f32]),
    "sa_score_phrase": (c_int, [P_void, P_u32, c_u32, c_u32, c_f32, c_f32, c_f32, c_f32, c_u64, c_u64, P_f32]),
    "sa_score_batch_topk": (c_int, [P_void, P_u32, P_u32, P_f32, c_u32, c_u32, c_f32, c_f32, c_f32, c_u32,
                                    P_u32, P_f32]),
    "sa_batch_upload": (c_int, [P_void, P_u32, P_u32, P_f32, c_u32, c_u32, c_f32, c_f32, c_f32, c_u32]),
    "sa_batch_execute": (c_int, [P_void]),
    "sa_batch_download": (c_int, [P_void, P_u32, P_f32, P_u32]),
    "sa_batch_row": (c_int, [P_void, c_u32, P_f32]),
    "sa_timer_start": (c_int, [P_void]),
    "sa_timer_stop": (c_int, [P_void, ctypes.POINTER(ctypes.c_double)]),
    "sa_stats_reset": (c_int, [P_void]),
    "sa_stats_get": (c_int, [P_void, ctypes.POINTER(SaStats)]),
    "sa_set_profiling": (c_int, [P_void, c_int]),
    "sa_comm_unique_id": (c_int, [P_void]),
    "sa_comm_init": (c_int, [P_void, P_void, c_int, c_int]),
    "sa_comm_destroy": (c_int, [P_void]),
    "sa_comm_barrier": (c_int, [P_void]),
    "sa_comm_allreduce_max": (c_int, [P_void, ctypes.POINTER(ctypes.c_double)]),
    "sa_comm_allreduce_sum_u64": (c_int, [P_void, P_u64, c_u64]),
    "sa_batch_execute_allgather": (c_int, [P_void]),
    "sa_batch_download_allgather": (c_int, [P_void, P_u32, P_f32, P_u32]),
    "sa_score_batch_topk_allgather": (c_int, [P_void, P_u32, P_u32, P_f32, c_u32, c_u32, c_f32, c_f32, c_f32,
                                              c_u32, P_u32, P_f32]),
    "sa_multi_create": (c_int, [ctypes.POINTER(P_void), c_u32, ctypes.POINTER(P_void)]),
    "sa_multi_destroy": (c_int, [P_void]),
    "sa_multi_qf": (c_int, [P_void, c_int, P_u32, P_u32, P_f32, P_f32, P_u32, P_f32, P_f32, P_f32, P_u32,
                            ctypes.c_double, P_u64]),
    "sa_multi_filter": (c_int, [P_void, c_u32, P_u32, c_u32, P_u64]),
    "sa_multi_phrases": (c_int, [P_void, c_u32, c_u32, P_u32, P_u32, P_u32, P_f32, c_f32, c_f32, c_f32]),
    "sa_multi_add_phase": (c_int, [P_void, c_u32, P_u32, P_u32, P_f32, P_u32]),
    "sa_multi_download": (c_int, [P_void, P_void, c_int]),
    "sa_multi_is_float32": (c_int, [P_void, ctypes.POINTER(c_int)]),
    "sa_multi_topk": (c_int, [P_void, c_u32, P_u32, ctypes.POINTER(ctypes.c_double)]),
    "sa_op_popcount64_reduce": (c_int, [P_u64, c_u64, c_int, P_u64, P_f32, P_u64]),
    "sa_op_bm25_score": (c_int, [P_f32, P_f32, c_u64, c_f32, c_f32, c_f32, c_f32, c_int]),
    "sa_op_similarity": (c_int, [c_int, P_f32, P_f32, c_u64, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                 ctypes.c_double, c_int, P_void]),
    "sa_op_bigram_freqs": (c_int, [P_u64, c_u64, P_u64, c_u64, c_int, c_int, P_u64, P_f32, P_u64, P_u64, P_u64]),
    "sa_op_intersect": (c_int, [P_u64, c_u64, P_u64, c_u64, c_u64, c_int, c_int, P_u64, P_u64, P_u64, P_u64]),
    "sa_op_adjacent": (c_int, [P_u64, c_u64, P_u64, c_u64, c_u64, c_int, P_u64, P_u64, P_u64]),
    "sa_op_intersect_with_adjacents": (c_int, [P_u64, c_u64, P_u64, c_u64, c_u64, c_int, P_u64, P_u64, P_u64,
                                               P_u64, P_u64, P_u64]),
    "sa_op_merge": (c_int, [P_u64, c_u64, P_u64, c_u64, c_int, c_int, P_u64, P_u64]),
    "sa_op_sort_merge_counts": (c_int, [P_u64, P_f32, c_u64, P_u64, P_f32, c_u64, c_int, P_u64, P_f32, P_u64]),
    "sa_op_unique": (c_int, [P_u64, c_u64, c_u64, c_int, P_u64, P_u64]),
    "sa_op_popcount64": (c_int, [P_u64, c_u64, c_int, P_u64]),
    "sa_op_popcount_reduce_at": (c_int, [P_u64, P_u64, c_u64, c_int, P_u64, P_f32, P_u64]),
    "sa_op_key_sum_over": (c_int, [P_u64, P_u64, c_u64, c_int, P_u64, P_f32, P_u64]),
    "sa_op_payload_slice": (c_int, [P_u64, c_u64, c_u64, c_u64, c_u64, c_int, P_u64, P_u64]),
    "sa_op_as_dense": (c_int, [P_u64, P_f32, c_u64, c_u64, c_int, P_f32]),
    "sa_op_last_staged_ctas": (c_u64, []),
    "sa_op_build_index": (c_int, [P_u32, P_u32, P_u32, c_u64, c_u32, c_int, P_u64, P_u64, P_u64, P_u64]),
}

_lib = None


class SearchArrayB200Error(RuntimeError):
    pass


def lib():
    """Loads the CUDA library; raises (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SearchArrayB200Error(
                f"{LIB_PATH} not found: build it with `python -m searcharray_b200.build` "
                "(there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)     # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().sa_last_error()
        raise SearchArrayB200Error(f"libsearcharray_b200 error {rc}: {msg.decode() if msg else ''}")


def p_u64(a):
    return a.ctypes.data_as(P_u64)


def p_u32(a):
    return a.ctypes.data_as(P_u32)


def p_f32(a):
    return a.ctypes.data_as(P_f32)
