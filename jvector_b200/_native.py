"""ctypes binding of libjvector_b200.so (the C ABI in include/jvector_b200.h). Fails loudly when the CUDA library is
missing or cannot be initialised: there is no CPU fallback in this package."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# JV_B200_SO: load a tuning variant of the library (tools/) instead of the product build
SO = os.environ.get("JV_B200_SO") or os.path.join(HERE, "lib", "libjvector_b200.so")

f32p = C.POINTER(C.c_float)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
u64p = C.POINTER(C.c_uint64)


class JVectorB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("jvector_b200 error %d: %s" % (code, msg))
        self.code = code


class SearchStats(C.Structure):
    _fields_ = [("visited", C.c_int64), ("expanded", C.c_int64), ("expanded_base", C.c_int64), ("reranked", C.c_int64),
                ("retried", C.c_int64), ("device_ms", C.c_double)]


class SearchOptions(C.Structure):
    _fields_ = [("accept_bits", C.c_void_p), ("accept_stride_words", C.c_int64), ("threshold", C.c_float), ("rerank_floor", C.c_float)]


class BuildParams(C.Structure):
    _fields_ = [("degree", C.c_int), ("beam_width", C.c_int), ("overflow", C.c_float), ("alpha", C.c_float),
                ("add_hierarchy", C.c_int), ("seed", C.c_uint64), ("max_batch", C.c_int), ("concurrent_window", C.c_int)]


# every symbol include/jvector_b200.h declares: (name, restype, argtypes)
_F, _I, _Z, _P, _L = C.c_float, C.c_int, C.c_size_t, C.c_void_p, C.c_int64
SYMBOLS = [
    # legacy libjvector.so ABI
    ("cosine_f32", _F, [f32p, _Z, f32p, _Z, _Z]), ("dot_product_f32", _F, [f32p, _Z, f32p, _Z, _Z]),
    ("euclidean_f32", _F, [f32p, _Z, f32p, _Z, _Z]), ("add_in_place_f32", None, [f32p, f32p, _Z]),
    ("add_scalar_in_place_f32", None, [f32p, _F, _Z]), ("sub_in_place_f32", None, [f32p, f32p, _Z]),
    ("sub_scalar_in_place_f32", None, [f32p, _F, _Z]), ("max_f32", _F, [f32p, _Z]), ("min_in_place_f32", None, [f32p, f32p, _Z]),
    ("assemble_and_sum_f32", _F, [f32p, _I, u8p, _I, _Z]), ("assemble_and_sum_pq_f32", _F, [f32p, _Z, u8p, _I, u8p, _I, _I]),
    ("pq_decoded_cosine_similarity_f32", _F, [u8p, _I, _Z, _I, f32p, f32p, _F]),
    ("calculate_partial_sums_dot_f32", None, [f32p, _I, _Z, _I, f32p, _I, f32p]),
    ("calculate_partial_sums_euclidean_f32", None, [f32p, _I, _Z, _I, f32p, _I, f32p]),
    ("calculate_partial_sums_self_magnitude_f32", None, [f32p, _I, _Z, _I, f32p]),
    ("nvq_quantize_8bit", None, [f32p, _Z, _F, _F, _F, _F, u8p]), ("nvq_loss", _F, [f32p, _Z, _F, _F, _F, _F, _I]),
    ("nvq_uniform_loss", _F, [f32p, _Z, _F, _F, _I]), ("nvq_square_l2_distance_8bit", _F, [f32p, u8p, _Z, _F, _F, _F, _F]),
    ("nvq_dot_product_8bit", _F, [f32p, u8p, _Z, _F, _F, _F, _F]),
    ("nvq_cosine_8bit_packed", _L, [f32p, u8p, _Z, _F, _F, _F, _F, f32p]), ("nvq_shuffle_query_in_place_8bit", None, [f32p, _Z]),
    ("jvector_simd_get_active_isa", C.c_char_p, []), ("jvector_simd_get_max_isa_env", C.c_char_p, []),
    # batched GPU ABI
    ("jv_gpu_init", _I, [_I]), ("jv_gpu_init_mask", _I, [C.c_uint32]), ("jv_gpu_bound_mask", C.c_uint32, []), ("jv_gpu_set_device", _I, [_I]),
    ("jv_gpu_device_count", _I, []), ("jv_last_error", C.c_char_p, []), ("jv_version", C.c_char_p, []),
    ("jv_gpu_sm_count", _I, []),
    ("jv_dataset_register_f32", _I, [f32p, _L, _I, C.POINTER(_P)]),
    ("jv_dataset_register_pq", _I, [u8p, _L, _I, _I, _I, f32p, f32p, C.POINTER(_P)]),
    ("jv_dataset_register_bq", _I, [u64p, _L, _I, C.POINTER(_P)]),
    ("jv_dataset_register_nvq", _I, [u8p, f32p, _L, _I, _I, f32p, C.POINTER(_P)]),
    ("jv_dataset_adopt_f32_device", _I, [_P, _L, _I, _I, C.POINTER(_P)]), ("jv_dataset_device", _I, [_P]),
    ("jv_dataset_invalidate_sketch", _I, [_P]), ("jv_dataset_f32_sketch", _I, [_P, C.POINTER(_I), C.POINTER(C.c_double), f32p, f32p, f32p]),
    ("jv_dataset_pq_pair_table", _I, [_P, _I]), ("jv_dataset_pq_pair_table_download", _I, [_P, _I, f32p]),
    ("jv_dataset_free", _I, [_P]), ("jv_dataset_size", _L, [_P]), ("jv_dataset_dim", _I, [_P]), ("jv_dataset_device_bytes", _L, [_P]),
    ("jv_query_begin", _I, [_P, f32p, _I, C.POINTER(_P)]), ("jv_score_batch", _I, [_P, i32p, _I, f32p]), ("jv_query_end", _I, [_P]),
    ("jv_query_get_lut", _I, [_P, f32p]),
    ("jv_query_batch_begin", _I, [_P, _I, f32p, _I, C.POINTER(_P)]), ("jv_query_batch_score", _I, [_P, i32p, i32p, f32p, C.POINTER(C.c_double)]),
    ("jv_query_batch_score_one", _I, [_P, _I, i32p, _I, f32p]), ("jv_query_batch_end", _I, [_P]),
    ("jv_score_multi", _I, [_P, _I, f32p, _I, i32p, i32p, f32p]), ("jv_score_pairs", _I, [_P, _I, i32p, i32p, _I, f32p]),
    ("jv_topk_bruteforce", _I, [_P, _I, f32p, _I, _I, i64p]),
    ("jv_topk_bruteforce_device", _I, [_P, _I, _P, _I, _I, _L, _P]), ("jv_topk_merge_device", _I, [_P, _I, _I, _I, _P]),
    ("jv_topk_bruteforce_device_async", _I, [_P, _I, _P, _I, _I, _L, _P, _P, _P]), ("jv_topk_merge_device_async", _I, [_P, _I, _I, _I, _P, _P]),
    ("jv_multi_register_bq", _I, [u64p, _L, _I, C.POINTER(_P)]), ("jv_multi_register_f32", _I, [f32p, _L, _I, C.POINTER(_P)]),
    ("jv_multi_free", _I, [_P]), ("jv_multi_shard_count", _I, [_P]), ("jv_multi_shard_info", _I, [_P, _I, C.POINTER(_I), i64p, i64p]),
    ("jv_multi_topk_bruteforce", _I, [_P, _I, f32p, _I, _I, i64p]),
    ("jv_multi_graph_search_batch", _I, [_I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _I, f32p, _I, _I, _I, C.POINTER(SearchOptions), i32p, f32p,
                                         C.POINTER(SearchStats)]),
    ("jv_bq_encode_batch", _I, [f32p, _L, _I, u64p]), ("jv_pq_encode_batch", _I, [f32p, _L, _I, _I, _I, f32p, f32p, u8p]),
    ("jv_nvq_encode_batch", _I, [f32p, _L, _I, _I, f32p, _I, f32p, u8p]),
    ("jv_kmeans_assign_batch", _I, [f32p, _L, _I, f32p, _I, i32p]),
    ("jv_bq_encode_dataset", _I, [_P, u64p]), ("jv_pq_encode_dataset", _I, [_P, _I, _I, f32p, f32p, u8p]),
    ("jv_nvq_encode_dataset", _I, [_P, _I, f32p, _I, f32p, u8p]),
    ("jv_nvq_encode_dataset_resident", _I, [_P, _I, f32p, _I, C.POINTER(_P)]),
    ("jv_graph_create", _I, [C.c_int32, _I, i32p, C.c_int32, C.POINTER(_P)]), ("jv_graph_add_level", _I, [_P, C.c_int32, i32p, i32p]),
    ("jv_graph_fuse_pq", _I, [_P, _P]), ("jv_graph_fused_download", _I, [_P, u8p, C.POINTER(_I)]),
    ("jv_graph_free", _I, [_P]), ("jv_graph_info", _I, [_P, i32p, C.POINTER(_I), C.POINTER(_I), i32p]),
    ("jv_graph_download", _I, [_P, _I, i32p, i32p, i32p]),
    ("jv_graph_search_batch", _I, [_P, _P, _P, _I, f32p, _I, _I, _I, i32p, f32p, C.POINTER(SearchStats)]),
    ("jv_graph_search_batch_device", _I, [_P, _P, _P, _I, _P, _I, _I, _I, _P, _P, C.POINTER(SearchStats)]),
    ("jv_graph_search_batch_ex", _I, [_P, _P, _P, _I, f32p, _I, _I, _I, C.POINTER(SearchOptions), i32p, f32p, C.POINTER(SearchStats)]),
    ("jv_graph_search_batch_device_ex", _I, [_P, _P, _P, _I, _P, _I, _I, _I, C.POINTER(SearchOptions), _P, _P, C.POINTER(SearchStats)]),
    ("jv_graph_build", _I, [_P, _I, C.POINTER(BuildParams), C.POINTER(_P), C.POINTER(C.c_double)]),
    ("jv_graph_build_stats", _I, [i64p, i64p, i64p]),
    ("jv_builder_create", _I, [_P, _I, C.POINTER(BuildParams), _P, C.POINTER(_P)]), ("jv_builder_info", _I, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    ("jv_builder_next_batch", _I, [_P, i32p, i32p]), ("jv_builder_insert_slice", _I, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    ("jv_builder_apply_new", _I, [_P, C.c_int32, C.c_int32, _P, _P, i32p]), ("jv_builder_reprune_slice", _I, [_P, C.c_int32, C.c_int32, _P, _P]),
    ("jv_builder_apply_repruned", _I, [_P, C.c_int32, _P, _P]), ("jv_builder_collect_over_degree", _I, [_P, i32p]),
    ("jv_builder_finish", _I, [_P, C.POINTER(_P), C.POINTER(C.c_double)]), ("jv_builder_free", _I, [_P]),
    ("jv_device_malloc", _I, [C.POINTER(_P), _Z]), ("jv_device_free", _I, [_P]), ("jv_memcpy_h2d", _I, [_P, _P, _Z]),
    ("jv_memcpy_d2h", _I, [_P, _P, _Z]), ("jv_host_register", _I, [_P, _Z]), ("jv_host_unregister", _I, [_P]),
    ("jv_device_synchronize", _I, []), ("jv_kernel_launch_count", _L, []), ("jv_search_rows_read", _L, []),
]

_lib = None
_inited = False


def load():
    """dlopen the library and bind every declared symbol (no CUDA call is made here)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        raise ImportError("jvector_b200: %s is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % SO)
    lib = C.CDLL(SO)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError here = ABI drift, fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise JVectorB200Error(rc, load().jv_last_error().decode())


def init(device=None):
    """Bind the process to a B200. Raises when no sm_100 device is present."""
    global _inited
    lib = load()
    if _inited:
        return lib
    if device is None:
        device = int(os.environ.get("JVECTOR_GPU_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    check(lib.jv_gpu_init(device))
    _inited = True
    return lib


def fp(a):
    return a.ctypes.data_as(f32p) if a is not None else None


def bp(a):
    return a.ctypes.data_as(u8p) if a is not None else None


def ip(a):
    return a.ctypes.data_as(i32p) if a is not None else None


def lp(a):
    return a.ctypes.data_as(i64p) if a is not None else None


def wp(a):
    return a.ctypes.data_as(u64p) if a is not None else None


def c32(a):
    return np.ascontiguousarray(a, dtype=np.float32)
