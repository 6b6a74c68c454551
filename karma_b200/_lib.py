"""ctypes binding of libkarma_b200.so (the C ABI in include/karma_b200.h).

There is deliberately no fallback: if the shared library is missing or a call
fails, a KarmaB200Error is raised.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkarma_b200.so")

KB_MODE_5P6 = 0
KB_MODE_DENSE_5_6 = 1
KB_MODE_DENSE_4_5 = 2
KB_KNN_AUTO, KB_KNN_SIMT, KB_KNN_TC = 0, 1, 2
KB_EINVAL, KB_ENOGPU, KB_EUNSUPPORTED = -1, -3, -4
KB_COUNT_NO_COLUMNS = 0x100

STAGES = {"count": 0, "count_long": 1, "compact": 2, "normalise": 3, "knn_gemm": 4, "rerank": 5, "knn_exact": 6, "readgraph": 7, "links": 8,
          "hdbscan_core": 9, "hdbscan_mst": 10, "hdbscan_sort": 11, "spectral_components": 12, "spectral_eigensolve": 13,
          "spectral_meta": 14, "mcl_setup": 15, "mcl_iteration": 16}


def KB_MODE_K(k):
    return 16 + int(k)


class KarmaB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libkarma_b200 error %d: %s" % (code, msg))
        self.code = code


# every symbol include/karma_b200.h declares: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    "kb_version": (c_int, []),
    "kb_last_error": (c_char_p, []),
    "kb_mode_columns": (c_int, [c_int]),
    "kb_create": (c_int, [POINTER(c_void_p), c_int]),
    "kb_destroy": (c_int, [_P]),
    "kb_set_stream": (c_int, [_P, _P]),
    "kb_count": (c_int, [_P, c_int, _P, _P, c_int64, _P, c_int64, _P, _P]),
    "kb_count_stats": (c_int, [_P, POINTER(c_int64), POINTER(c_int64)]),
    "kb_exotic_collect": (c_int, [_P, c_int, _P, _P, c_int64, _P, POINTER(c_int64), POINTER(c_int64)]),
    "kb_exotic_fetch": (c_int, [_P, _P, _P, _P, _P]),
    "kb_exotic_scatter": (c_int, [_P, _P, _P, c_int64]),
    "kb_kmer_sorted_collect": (c_int, [_P, c_int, _P, _P, c_int64, POINTER(c_int64), POINTER(c_int64)]),
    "kb_kmer_sorted_fetch": (c_int, [_P, _P, _P]),
    "kb_compact": (c_int, [_P, _P, c_int64, c_int32, _P, c_int64, _P, c_int64, c_int32]),
    "kb_normalise": (c_int, [_P, _P, c_int64, c_int32, _P, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, _P, _P]),
    "kb_count_profile": (c_int, [_P, c_int, _P, _P, _P, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, _P, _P, _P]),
    "kb_rowmeta_flags_or": (c_int, [_P, _P, c_int64, _P]),
    "kb_knn_workspace_bytes": (c_int64, [_P, c_int64, c_int64, c_int64, c_int32, c_int32, c_int, c_int64]),
    "kb_knn": (c_int, [_P, c_int, c_int32, _P, c_int64, c_int32, _P, c_int64, c_int64, c_int64,
                       _P, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64, _P]),
    "kb_knn_fixup": (c_int64, [_P, c_int, c_int32, _P, c_int64, c_int32, _P, c_int64, c_int64, c_int64,
                               _P, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64]),
    "kb_knn_uncertified_ptr": (c_int, [_P, c_int64, c_int64, c_int64, c_int32, c_int32, c_int, c_int64, _P, POINTER(c_void_p)]),
    "kb_knn_plan_info": (c_int, [c_int, c_int, c_int64, c_int64, c_int64, c_int32, c_int32, POINTER(c_int64)]),
    "kb_knn_plan_table": (c_int, [c_int, c_int, c_int64, c_int64, c_int64, c_int32, c_int32, _P, _P, _P]),
    "kb_xchg_create": (c_int, [_P, c_int, c_int, c_int64, POINTER(c_void_p), POINTER(c_void_p), _P]),
    "kb_xchg_attach": (c_int, [_P, _P]),
    "kb_xchg_peer_ptr": (c_int, [_P, c_int, POINTER(c_void_p)]),
    "kb_xchg_flags": (c_int, [_P, POINTER(c_void_p), POINTER(c_void_p)]),
    "kb_xchg_destroy": (c_int, [_P]),
    "kb_xchg_warm": (c_int, [_P, c_int, _P, _P]),
    "kb_xchg_begin": (c_int, [_P]),
    "kb_xchg_push": (c_int, [_P, _P, c_int, _P, _P]),
    "kb_xchg_finish": (c_int, [_P, c_int64, c_int32]),
    "kb_fasta_open": (c_int, [c_char_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
    "kb_fasta_fill": (c_int, [_P, _P, _P, _P, _P, _P]),
    "kb_fasta_close": (c_int, [_P]),
    "kb_eq_open": (c_int, [c_char_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
    "kb_eq_fill": (c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "kb_eq_close": (c_int, [_P]),
    "kb_readgraph_build": (c_int, [_P, c_int64, c_int64, _P, _P, _P, _P, _P, POINTER(c_int64)]),
    "kb_readgraph_fetch": (c_int, [_P, _P, _P, _P, _P]),
    "kb_links_build": (c_int, [_P, c_int64, _P, _P, _P, c_int64, _P, _P, _P, _P, c_int64, c_int64, c_double, POINTER(c_int64)]),
    "kb_links_fetch": (c_int, [_P, _P, _P, _P, _P, _P]),
    "kb_fuzzy_graph_build": (c_int, [_P, c_int64, c_int32, _P, _P, c_double, c_double, _P, _P, POINTER(c_int64)]),
    "kb_fuzzy_graph_fetch": (c_int, [_P, _P, _P, _P]),
    "kb_umap_layout": (c_int, [_P, c_int64, c_int64, _P, _P, _P, c_int32, c_int32, c_double, c_double, c_double, c_double, c_double,
                               c_uint64, _P, _P, POINTER(c_int64)]),
    "kb_hdbscan_mst": (c_int, [_P, c_int64, c_int32, _P, c_int32, _P, _P, _P]),
    "kb_hdbscan_labels": (c_int, [c_int64, _P, _P, c_int32, c_int32, _P, _P, POINTER(c_int64)]),
    "kb_spectral_build": (c_int, [_P, c_int64, c_int64, _P, _P, _P, c_int32, c_int32, _P, c_int32, c_int64, POINTER(c_int64)]),
    "kb_spectral_fetch": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "kb_spectral_assemble": (c_int, [_P, _P, _P]),
    "kb_mcl_build": (c_int, [_P, c_int64, c_int64, _P, _P, _P, _P, c_int64, c_double, POINTER(c_int64), POINTER(c_int64)]),
    "kb_mcl_fetch": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "kb_enable_timing": (c_int, [_P, c_int]),
    "kb_stage_ms": (c_int, [_P, c_int, POINTER(c_float), POINTER(c_int)]),
    "kb_launch_count": (c_int64, [_P]),
}

_lib = None


def load():
    """Load the shared library (build it first with ``python -m karma_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KarmaB200Error(-100, "%s not found: run `python -m karma_b200.build` "
                             "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc < 0:
        raise KarmaB200Error(rc, load().kb_last_error().decode("utf-8", "replace"))
    return rc


def ptr(t):
    """data_ptr of a torch tensor (or None)."""
    return None if t is None else c_void_p(t.data_ptr())
