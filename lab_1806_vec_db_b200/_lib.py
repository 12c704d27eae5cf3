"""ctypes loader for libvdb_b200.so (the C ABI in include/vdb_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or a call fails, this raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VDB_LIB_PATH") or os.path.join(_HERE, "libvdb_b200.so")

OK, EINVAL, ECUDA, ENOMEM, EUNSUPPORTED = 0, 1, 2, 3, 4
L2SQR, COSINE, DOT = 0, 1, 2
F32, U8 = 0, 1


class VdbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vdb_b200 error {code}: {msg}")
        self.code = code


_lib = None

u32, u64, i32, f32, vp = C.c_uint32, C.c_uint64, C.c_int, C.c_float, C.c_void_p

# name -> (restype, argtypes); every symbol declared in include/vdb_b200.h is listed here
SIGNATURES = {
    "vdb_last_error": (C.c_char_p, []),
    "vdb_version": (i32, []),
    "vdb_device_count": (i32, [vp]),
    "vdb_set_device": (i32, [i32]),
    "vdb_init": (i32, [vp, u32]),
    "vdb_dataset_create_sharded_dev": (i32, [vp, vp, vp, u32, u32, u32, i32, i32, u64, vp]),
    "vdb_dataset_shards": (i32, [vp, vp]),
    "vdb_dataset_shard": (i32, [vp, u32, vp, vp, vp, vp]),
    "vdb_dataset_set_flat_path": (i32, [vp, i32]),
    "vdb_flat_knn_sharded_dev": (i32, [vp, vp, u32, u32, vp, vp, vp]),
    "vdb_debug_force_redo": (i32, [u32]),
    "vdb_dataset_create": (i32, [vp, u64, u32, i32, i32, u64, vp]),
    "vdb_dataset_create_dev": (i32, [vp, u64, u32, u32, i32, i32, u64, vp]),
    "vdb_dataset_append": (i32, [vp, vp, u64]),
    "vdb_dataset_swap_remove": (i32, [vp, u64]),
    "vdb_dataset_len": (i32, [vp, vp]),
    "vdb_dataset_dim": (i32, [vp, vp]),
    "vdb_dataset_destroy": (i32, [vp]),
    "vdb_calc_dist": (i32, [vp, vp, u64, u32, i32, i32, vp]),
    "vdb_row_cache": (i32, [vp, vp]),
    "vdb_gather_dist": (i32, [vp, vp, u32, vp, vp, vp]),
    "vdb_flat_knn": (i32, [vp, vp, u32, u32, vp, vp, vp]),
    "vdb_flat_knn_dev": (i32, [vp, vp, u32, u32, vp, vp, vp, vp]),
    "vdb_flat_knn_keys_dev": (i32, [vp, vp, u32, u32, vp, vp]),
    "vdb_merge_keys_dev": (i32, [vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_flat_set_path": (i32, [i32]),
    "vdb_set_batching": (i32, [i32]),
    "vdb_parallel_knn": (i32, [vp, vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_batch_stats": (i32, [vp, vp, vp]),
    "vdb_kmeans_assign": (i32, [vp, u64, u32, i32, i32, vp, u32, u32, u32, vp]),
    "vdb_kmeans_assign_ds": (i32, [vp, vp, u32, u32, u32, vp]),
    "vdb_kmeans_train": (i32, [vp, u64, u32, i32, i32, vp, u32, u32, u32, u32, f32, vp]),
    "vdb_kmeans_train_ds": (i32, [vp, vp, u32, u32, u32, u32, f32, vp]),
    "vdb_kmeans_pp_init_ds": (i32, [vp, u32, u32, u32, vp, vp]),
    "vdb_kmeans_pp_weights": (i32, [vp, u64, u32, i32, i32, vp, u32, u32, vp]),
    "vdb_pq_groups": (i32, [u32, u32, vp]),
    "vdb_pq_create": (i32, [vp, vp, u32, u32, vp, vp]),
    "vdb_pq_create_from_codes": (i32, [vp, vp, u32, u32, vp, vp]),
    "vdb_pq_destroy": (i32, [vp]),
    "vdb_pq_lut": (i32, [vp, vp, u32, vp, vp]),
    "vdb_pq_adc_all": (i32, [vp, vp, u32, vp]),
    "vdb_pq_knn": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp]),
    "vdb_pq_knn_dev": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_pq_adc_keys_dev": (i32, [vp, vp, vp, u32, u32, vp, vp]),
    "vdb_pq_rerank_keys_dev": (i32, [vp, vp, u32, vp, u32, u32, vp, vp]),
    "vdb_ivf_knn_keys_dev": (i32, [vp, vp, vp, u32, u32, u32, vp, vp]),
    "vdb_ivf_create": (i32, [vp, vp, u32, vp, vp]),
    "vdb_ivf_destroy": (i32, [vp]),
    "vdb_pq_train_ds": (i32, [vp, u32, u32, u32, f32, vp, vp, vp, vp]),
    "vdb_hnsw_build": (i32, [vp, u32, u32, vp, u32, vp]),
    "vdb_hnsw_destroy": (i32, [vp]),
    "vdb_hnsw_append": (i32, [vp, vp, vp, u32]),
    "vdb_hnsw_info": (i32, [vp, vp, vp, vp, vp, vp]),
    "vdb_hnsw_links0": (i32, [vp, vp, vp]),
    "vdb_hnsw_overflow": (i32, [vp, vp]),
    "vdb_hnsw_evals": (i32, [vp, vp, i32]),
    "vdb_hnsw_upper": (i32, [vp, vp, vp, vp]),
    "vdb_hnsw_create_from_graph": (i32, [vp, u32, u32, vp, vp, vp, vp, vp, C.c_int64, C.c_int32, vp]),
    "vdb_hnsw_knn": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp]),
    "vdb_hnsw_knn_dev": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_hnsw_knn_pq": (i32, [vp, vp, vp, vp, u32, u32, u32, vp, vp, vp]),
    "vdb_hnsw_knn_pq_dev": (i32, [vp, vp, vp, vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_ivf_lists": (i32, [vp, vp, vp]),
    "vdb_ivf_knn": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp]),
    "vdb_ivf_knn_dev": (i32, [vp, vp, vp, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_ivf_knn_pq": (i32, [vp, vp, vp, vp, u32, u32, u32, u32, vp, vp, vp]),
    "vdb_ivf_knn_pq_dev": (i32, [vp, vp, vp, vp, u32, u32, u32, u32, vp, vp, vp, vp]),
    "vdb_ivf_pq_adc_keys_dev": (i32, [vp, vp, vp, vp, u32, u32, u32, vp, vp]),
    "vdb_tq_info": (i32, [vp, vp, vp, vp, vp]),
    "vdb_tq_j0": (u32, [u32, u64, u64]),
    "vdb_tq_begin_dev": (i32, [vp, vp, u32, vp, vp]),
    "vdb_tq_sample_dev": (i32, [vp, u32, vp]),
    "vdb_tq_tau_dev": (i32, [vp, vp, u32, u32, u32, vp]),
    "vdb_tq_sample_j": (u32, [u32, u64]),
    "vdb_tq_filter_dev": (i32, [vp, u32, vp, vp, vp]),
    "vdb_tq_check_dev": (i32, [vp, vp, u32, u64, vp, vp, vp, vp]),
    "vdb_tq_end": (i32, [vp]),
    "vdb_flat_scan_keys_dev": (i32, [vp, vp, u32, u32, vp, vp]),
    "vdb_merge_keys_to_keys_dev": (i32, [vp, u32, u32, u32, vp, vp]),
    "vdb_decode_keys_dev": (i32, [vp, u32, u32, vp, vp, vp, vp]),
    "vdb_debug_gemm_scores_dev": (i32, [vp, vp, u32, u32, i32, vp, vp]),
    "vdb_debug_pq_bounds_dev": (i32, [vp, vp, u32, i32, vp, vp, vp]),
    "vdb_dataset_operand_info": (i32, [vp, vp, vp, vp, vp, vp]),
    "vdb_dataset_drop_side_arrays": (i32, [vp]),
    "vdb_flat_gemm_fallbacks": (u64, []),
    "vdb_flat_gemm_stats": (i32, [vp, vp, vp]),
    "vdb_launch_count": (u64, []),
    "vdb_prof_enable": (i32, [i32]),
    "vdb_prof_reset": (i32, []),
    "vdb_prof_read": (i32, [C.c_char_p, vp, vp]),
}


def lib():
    """Loads the CUDA library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C lab_1806_vec_db_b200/csrc`. There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise VdbError(rc, lib().vdb_last_error().decode("utf-8", "replace"))


def ptr(a):
    """void* of a numpy array (must be C-contiguous) or a raw integer device pointer."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def metric_code(dist):
    """Metric names follow the pyo3 layer (reference src/pyo3/mod.rs:15-22)."""
    if isinstance(dist, str):
        d = dist.lower()
        if d == "l2sqr":
            return L2SQR
        if d == "cosine":
            return COSINE
        raise ValueError(f"Invalid distance function: {dist}")
    return int(dist)


def dtype_code(a):
    if a.dtype == np.float32:
        return F32
    if a.dtype == np.uint8:
        return U8
    raise TypeError(f"unsupported scalar type {a.dtype}; the reference supports f32 and u8 (src/scalar.rs:117-119)")
