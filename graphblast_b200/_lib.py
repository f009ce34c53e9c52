"""ctypes loader for libgraphblast_b200.so (the C ABI in include/graphblast_b200.h).

The product path fails loudly when the CUDA extension is missing: there is no CPU
fallback and nothing under oracle/ is ever imported from here.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GB200_LIB: another build of the same library (kernel-parameter experiments)
LIB_PATH = os.environ.get("GB200_LIB") or os.path.join(_HERE, "lib", "libgraphblast_b200.so")

_lib = None

# (name, restype, argtypes) for every symbol declared in include/graphblast_b200.h
_P = C.c_void_p
_I = C.c_int
_IP = C.POINTER(C.c_int)
_D = C.c_double
_F = C.c_float
_LL = C.c_longlong
_ULL = C.c_ulonglong
_S = C.c_char_p

SIGNATURES = [
    ("gb200_init", _I, [_I]),
    ("gb200_set_stream", _I, [_P]),
    ("gb200_sync", _I, []),
    ("gb200_sm_count", _I, [_IP]),
    ("gb200_version", _S, []),
    ("gb200_desc_new", _I, [C.POINTER(_P)]),
    ("gb200_desc_free", _I, [_P]),
    ("gb200_desc_set", _I, [_P, _I, _I]),
    ("gb200_desc_get", _I, [_P, _I, _IP]),
    ("gb200_desc_toggle", _I, [_P, _I]),
    ("gb200_desc_set_knob", _I, [_P, _S, _D]),
    ("gb200_desc_get_knob", _I, [_P, _S, C.POINTER(_D)]),
    ("gb200_matrix_new", _I, [C.POINTER(_P), _I, _I, _I]),
    ("gb200_matrix_free", _I, [_P]),
    ("gb200_matrix_build_coo", _I, [_P, _P, _P, _P, _I, _I]),
    ("gb200_matrix_load_mtx", _I, [C.POINTER(_P), _I, _S, _I]),
    ("gb200_matrix_adopt_csr", _I, [_P, _P, _P, _P, _I]),
    ("gb200_matrix_build_coo_device", _I, [_P, _P, _P, _P, _LL, _I]),
    ("gb200_ingest_coo", _I, [_I, _I, _P, _P, _P, _LL, _I, C.POINTER(_P),
                              C.POINTER(_LL)]),
    ("gb200_ingest_export", _I, [_P, _P, _P, _P]),
    ("gb200_ingest_free", _I, [_P]),
    ("gb200_csr_transpose_values", _I, [_I, _I, _I, _P, _P, _P, _P, _P, _P]),
    ("gb200_sort_pairs_u64", _I, [_P, _P, _LL, _I]),
    ("gb200_matrix_adopt_csc", _I, [_P, _P, _P, _P, _I]),
    ("gb200_matrix_nrows", _I, [_P, _IP]),
    ("gb200_matrix_ncols", _I, [_P, _IP]),
    ("gb200_matrix_nvals", _I, [_P, _IP]),
    ("gb200_matrix_extract_csr", _I, [_P, _P, _P, _P]),
    ("gb200_matrix_tril", _I, [_P, _P]),
    ("gb200_matrix_apply_uniform_random", _I, [_P, _P, _I, _I, _I]),
    ("gb200_host_uniform_weights", _I, [_I, _I, _I, _LL, _P]),
    ("gb200_pr_normalize", _I, [_P, _F, _P]),
    ("gb200_vector_new", _I, [C.POINTER(_P), _I, _I]),
    ("gb200_vector_free", _I, [_P]),
    ("gb200_vector_fill", _I, [_P, _D]),
    ("gb200_vector_build_sparse", _I, [_P, _P, _P, _I]),
    ("gb200_vector_build_dense", _I, [_P, _P, _I]),
    ("gb200_vector_adopt_dense", _I, [_P, _P, _I]),
    ("gb200_vector_adopt_sparse", _I, [_P, _P, _P, _I]),
    ("gb200_vector_set_element", _I, [_P, _D, _I]),
    ("gb200_vector_size", _I, [_P, _IP]),
    ("gb200_vector_nvals", _I, [_P, _IP]),
    ("gb200_vector_storage", _I, [_P, _IP]),
    ("gb200_vector_extract_dense", _I, [_P, _P, _I]),
    ("gb200_vector_extract_sparse", _I, [_P, _P, _P, _IP]),
    ("gb200_vector_swap", _I, [_P, _P]),
    ("gb200_vector_dup", _I, [_P, _P]),
    ("gb200_vector_clear", _I, [_P]),
    ("gb200_vector_sparse2dense", _I, [_P, _D, _P]),
    ("gb200_vector_dense2sparse", _I, [_P, _D, _P]),
    ("gb200_vector_device_ptr", _I, [_P, C.POINTER(_P)]),
    ("gb200_vxm", _I, [_P, _P, _I, _I, _P, _P, _P]),
    ("gb200_mxv", _I, [_P, _P, _I, _I, _P, _P, _P]),
    ("gb200_mxm", _I, [_P, _P, _I, _P, _P, _P]),
    ("gb200_ewise_add", _I, [_P, _P, _I, _P, _P, _P]),
    ("gb200_ewise_add_scalar", _I, [_P, _P, _I, _P, _D, _P]),
    ("gb200_ewise_mult", _I, [_P, _P, _I, _P, _P, _P]),
    ("gb200_assign_scalar", _I, [_P, _P, _D, _P]),
    ("gb200_reduce_vector", _I, [C.POINTER(_D), _I, _P, _P]),
    ("gb200_reduce_matrix", _I, [C.POINTER(_D), _I, _P, _P]),
    ("gb200_reduce_matrix_rows", _I, [_P, _I, _P, _P]),
    ("gb200_bfs", _I, [_P, _P, _I, _P, C.POINTER(_F)]),
    ("gb200_bfs_stats", _I, [_P, _I, _P]),
    ("gb200_scatter", _I, [_P, _P, _F, _P]),
    ("gb200_assign_scatter", _I, [_P, _P, _P, _P]),
    ("gb200_extract_gather", _I, [_P, _P, _P, _P]),
    ("gb200_sssp", _I, [_P, _P, _I, _P, C.POINTER(_F)]),
    ("gb200_pr", _I, [_P, _P, _F, _F, _P, C.POINTER(_F)]),
    ("gb200_tc", _I, [C.POINTER(_LL), _P, _P, _P, C.POINTER(_F)]),
    ("gb200_rmat_edges", _I, [_I, _LL, _ULL, _LL, _P, _P]),
    ("gb200_vector_export_bits", _I, [_P, _P, C.POINTER(_LL)]),
    ("gb200_vector_export_bits_async", _I, [_P, _P, _P]),
    ("gb200_vector_import_bits", _I, [_P, _P, _LL]),
    ("gb200_profile_enable", _I, [_I]),
    ("gb200_profile_reset", _I, []),
    ("gb200_profile_read", _I, [_I, C.POINTER(_D), C.POINTER(_LL),
                                C.POINTER(_D)]),
    ("gb200_launch_count", _I, [C.POINTER(_ULL)]),
    ("gb200_xchg_create", _I, [C.POINTER(_P), _I, _I, C.POINTER(_LL)]),
    ("gb200_xchg_handle", _I, [_P, _P]),
    ("gb200_xchg_connect", _I, [_P, _P]),
    ("gb200_xchg_free", _I, [_P]),
    ("gb200_xchg_allgather_bits", _I, [_P, _P, C.POINTER(_LL)]),
    ("gb200_xchg_bits_ptr", _I, [_P, C.POINTER(_P)]),
    ("gb200_dist_bfs_fused", _I, [_P, _P, _P, _LL, _LL, _P, C.POINTER(_I)]),
    ("gb200_xchg_allgather_words", _I, [_P, _P, _D, C.POINTER(_D)]),
    ("gb200_dist_pr", _I, [_P, _P, _P, _LL, _F, _F, _P, C.POINTER(_I)]),
    ("gb200_dist_sssp", _I, [_P, _P, _P, _LL, _LL, _P, C.POINTER(_I)]),
]


class ExtensionMissing(RuntimeError):
    pass


def load():
    """Loads the shared library; raises ExtensionMissing (never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ExtensionMissing(
            "graphblast_b200: %s not found. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SIGNATURES:
        fn = getattr(lib, name)   # AttributeError if a declared symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib
