"""ctypes image of include/spmv_b200.h (the C ABI of libspmv_b200.so).

Only struct layouts and prototypes live here -- no logic.  Every Structure
mirrors one POD struct of the header (and therefore one struct of the
reference API, file:line cited in the header).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SPMV_B200_LIB: another build of the same library (A/B timing of build-time constants)
LIB_PATH = os.environ.get("SPMV_B200_LIB") or os.path.join(_HERE, "lib", "libspmv_b200.so")

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)
c_double_p = C.POINTER(C.c_double)
c_uint32_p = C.POINTER(C.c_uint32)


class CSRMatrix(C.Structure):  # spmv_b200_csr == spmv::CSRMatrix (72 B)
    _fields_ = [
        ("num_rows", C.c_int), ("num_cols", C.c_int), ("nnz", C.c_int),
        ("values", c_float_p), ("col_indices", c_int_p), ("row_ptrs", c_int_p),
        ("d_values", C.c_void_p), ("d_col_indices", C.c_void_p), ("d_row_ptrs", C.c_void_p),
        ("owns_host_memory", C.c_bool), ("owns_device_memory", C.c_bool),
    ]


class ELLMatrix(C.Structure):  # spmv_b200_ell == spmv::ELLMatrix (56 B)
    _fields_ = [
        ("num_rows", C.c_int), ("num_cols", C.c_int), ("max_nnz_per_row", C.c_int),
        ("values", c_float_p), ("col_indices", c_int_p),
        ("d_values", C.c_void_p), ("d_col_indices", C.c_void_p),
        ("owns_host_memory", C.c_bool), ("owns_device_memory", C.c_bool),
    ]


class CSRStats(C.Structure):
    _fields_ = [("avg_nnz_per_row", C.c_float), ("max_nnz_per_row", C.c_int),
                ("min_nnz_per_row", C.c_int), ("skewness", C.c_float)]


class SpMVConfig(C.Structure):
    _fields_ = [("kernel_type", C.c_int), ("block_size", C.c_int), ("use_texture", C.c_bool)]


class SpMVResult(C.Structure):
    _fields_ = [("y", C.c_void_p), ("elapsed_ms", C.c_float), ("gflops", C.c_float),
                ("bandwidth_gb_s", C.c_float), ("error_code", C.c_int)]


class BandwidthMetrics(C.Structure):
    _fields_ = [("theoretical_bandwidth_gb_s", C.c_float), ("achieved_bandwidth_gb_s", C.c_float),
                ("efficiency", C.c_float)]


class PageRankConfig(C.Structure):
    _fields_ = [("damping_factor", C.c_float), ("tolerance", C.c_float), ("max_iterations", C.c_int)]


class PageRankResult(C.Structure):
    _fields_ = [("ranks", c_float_p), ("iterations", C.c_int), ("final_residual", C.c_float),
                ("converged", C.c_bool)]


class TopKNode(C.Structure):
    _fields_ = [("node_id", C.c_int), ("rank", C.c_float)]


class BenchmarkConfig(C.Structure):
    _fields_ = [("num_warmup_runs", C.c_int), ("num_runs", C.c_int), ("compare_cpu", C.c_bool)]


class BenchmarkResult(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("execution_time_ms", C.c_float), ("gflops", C.c_float),
                ("bandwidth_gb_s", C.c_float), ("avg_time_ms", C.c_float), ("min_time_ms", C.c_float),
                ("max_time_ms", C.c_float), ("stddev_time_ms", C.c_float), ("num_runs", C.c_int)]


CSR_P = C.POINTER(CSRMatrix)
ELL_P = C.POINTER(ELLMatrix)
CFG_P = C.POINTER(SpMVConfig)
RES_P = C.POINTER(SpMVResult)
PRC_P = C.POINTER(PageRankConfig)
PRR_P = C.POINTER(PageRankResult)
BC_P = C.POINTER(BenchmarkConfig)
BR_P = C.POINTER(BenchmarkResult)
vp = C.c_void_p

# name -> (restype, argtypes); the complete list of symbols include/spmv_b200.h declares
PROTOTYPES = {
    "spmv_b200_error_string": (C.c_char_p, [C.c_int]),
    # A. CSR
    "spmv_b200_csr_create": (CSR_P, [C.c_int, C.c_int, C.c_int]),
    "spmv_b200_csr_destroy": (None, [CSR_P]),
    "spmv_b200_csr_from_dense": (C.c_int, [CSR_P, c_float_p, C.c_int, C.c_int]),
    "spmv_b200_csr_to_dense": (C.c_int, [CSR_P, c_float_p]),
    "spmv_b200_csr_get_element": (C.c_float, [CSR_P, C.c_int, C.c_int]),
    "spmv_b200_csr_to_gpu": (C.c_int, [CSR_P]),
    "spmv_b200_csr_from_gpu": (C.c_int, [CSR_P]),
    "spmv_b200_csr_free_gpu": (None, [CSR_P]),
    "spmv_b200_csr_serialize": (C.c_int, [CSR_P, C.c_char_p]),
    "spmv_b200_csr_deserialize": (C.c_int, [CSR_P, C.c_char_p]),
    "spmv_b200_csr_compute_stats": (C.c_int, [CSR_P, C.POINTER(CSRStats)]),
    # B. ELL
    "spmv_b200_ell_create": (ELL_P, [C.c_int, C.c_int, C.c_int]),
    "spmv_b200_ell_destroy": (None, [ELL_P]),
    "spmv_b200_ell_from_dense": (C.c_int, [ELL_P, c_float_p, C.c_int, C.c_int]),
    "spmv_b200_ell_from_csr": (C.c_int, [ELL_P, CSR_P]),
    "spmv_b200_ell_to_dense": (C.c_int, [ELL_P, c_float_p]),
    "spmv_b200_ell_get_element": (C.c_float, [ELL_P, C.c_int, C.c_int]),
    "spmv_b200_ell_to_gpu": (C.c_int, [ELL_P]),
    "spmv_b200_ell_from_gpu": (C.c_int, [ELL_P]),
    "spmv_b200_ell_free_gpu": (None, [ELL_P]),
    "spmv_b200_ell_serialize": (C.c_int, [ELL_P, C.c_char_p]),
    "spmv_b200_ell_deserialize": (C.c_int, [ELL_P, C.c_char_p]),
    "spmv_b200_ell_index": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    # C. SpMV
    "spmv_b200_spmv_cpu_csr": (None, [CSR_P, c_float_p, c_float_p]),
    "spmv_b200_spmv_cpu_ell": (None, [ELL_P, c_float_p, c_float_p]),
    "spmv_b200_spmv_csr": (C.c_int, [CSR_P, vp, vp, CFG_P, C.c_int, RES_P]),
    "spmv_b200_spmv_ell": (C.c_int, [ELL_P, vp, vp, CFG_P, C.c_int, RES_P]),
    "spmv_b200_auto_config": (C.c_int, [CSR_P, CFG_P]),
    "spmv_b200_validate_dimensions": (C.c_bool, [C.c_int, C.c_int]),
    # D. bandwidth / PageRank / benchmark
    "spmv_b200_bandwidth_csr": (C.c_int, [CSR_P, C.c_float, C.POINTER(BandwidthMetrics)]),
    "spmv_b200_bandwidth_ell": (C.c_int, [ELL_P, C.c_float, C.POINTER(BandwidthMetrics)]),
    "spmv_b200_peak_bandwidth": (C.c_float, []),
    "spmv_b200_pagerank": (C.c_int, [CSR_P, PRC_P, PRR_P]),
    "spmv_b200_pagerank_free": (None, [PRR_P]),
    "spmv_b200_pagerank_top_k": (C.c_int, [PRR_P, C.c_int, C.c_int, C.POINTER(TopKNode)]),
    "spmv_b200_benchmark_csr": (C.c_int, [CSR_P, c_float_p, CFG_P, BC_P, BR_P]),
    "spmv_b200_benchmark_ell": (C.c_int, [ELL_P, c_float_p, BC_P, BR_P]),
    "spmv_b200_compare_gpu_cpu_csr": (C.c_int, [CSR_P, c_float_p, CFG_P, BC_P, BR_P, BR_P, c_float_p]),
    "spmv_b200_benchmark_to_json": (C.c_int, [BR_P, C.c_char_p, C.c_int]),
    "spmv_b200_benchmark_from_json": (C.c_int, [C.c_char_p, BR_P]),
    "spmv_b200_benchmark_csr_report": (C.c_int, [CSR_P, c_float_p, CFG_P, BC_P, C.c_float, C.c_char_p, C.c_int]),
    # E. extensions
    "spmv_b200_version": (C.c_char_p, []),
    "spmv_b200_set_l2_fetch_granularity": (C.c_int, [C.c_int]),
    "spmv_b200_get_l2_fetch_granularity": (C.c_int, []),
    "spmv_b200_l2_persistence_limits": (C.c_int, [C.POINTER(C.c_ulonglong)] * 3),
    "spmv_b200_set_l2_persistence": (C.c_int, [vp, vp, C.c_ulonglong, C.c_float, C.c_ulonglong]),
    "spmv_b200_launch_count": (C.c_ulonglong, []),
    "spmv_b200_reference_policy": (C.c_int, [CSR_P, CFG_P]),
    "spmv_b200_spmv_csr_async": (C.c_int, [CSR_P, vp, vp, CFG_P, vp]),
    "spmv_b200_spmv_ell_async": (C.c_int, [ELL_P, vp, vp, vp]),
    "spmv_b200_pagerank_multi": (C.c_int, [CSR_P, vp, C.c_int, c_int_p, C.c_int, C.c_int, C.c_int, vp, vp]),
    "spmv_b200_comm_create": (C.c_int, [C.c_int, C.c_int, C.c_char_p, C.c_int, C.POINTER(vp)]),
    "spmv_b200_comm_destroy": (None, [vp]),
    "spmv_b200_comm_barrier": (C.c_int, [vp]),
    "spmv_b200_comm_allgather": (C.c_int, [vp, vp, vp, C.c_size_t]),
    "spmv_b200_comm_allgather_fds": (C.c_int, [vp, C.c_int, c_int_p]),
    "spmv_b200_pr_dist_create": (C.c_int, [vp, CSR_P, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "spmv_b200_pr_dist_run": (C.c_int, [vp, vp, C.c_int, vp]),
    "spmv_b200_pr_dist_ranks": (vp, [vp]),
    "spmv_b200_pr_dist_exchange": (C.c_int, [vp]),
    "spmv_b200_pr_dist_hub_columns": (C.c_int, [vp]),
    "spmv_b200_pr_dist_destroy": (None, [vp]),
    "spmv_b200_nccl_available": (C.c_int, []),
    "spmv_b200_ell_host_plan_create": (C.c_int, [ELL_P, C.c_int, C.POINTER(vp)]),
    "spmv_b200_ell_host_plan_destroy": (None, [vp]),
    "spmv_b200_spmv_ell_host": (C.c_int, [vp, vp, vp]),
    "spmv_b200_ell_host_plan_info": (C.c_int, [vp, c_int_p, c_int_p, c_int_p]),
    "spmv_b200_ell_host_plan_gated": (C.c_int, [vp, c_int_p, c_int_p]),
    "spmv_b200_probe_h2d_order": (C.c_int, [vp, C.c_ulonglong, C.c_int, C.POINTER(C.c_longlong), C.c_int, C.c_uint]),
    "spmv_b200_ell_host_plan_bytes": (C.c_int, [vp, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "spmv_b200_ell_from_csr_device": (C.c_int, [ELL_P, CSR_P]),
    "spmv_b200_merge_path_search": (C.c_int, [C.c_int, c_int_p, C.c_int, C.c_int, c_int_p, c_int_p]),
    "spmv_b200_partition_rows": (C.c_int, [c_int_p, C.c_int, C.c_int, c_int_p]),
    "spmv_b200_partition_rows_weighted": (C.c_int, [c_int_p, C.c_int, C.c_int, C.c_int, c_int_p]),
    "spmv_b200_pagerank_top_k_device": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(TopKNode)]),
    "spmv_b200_csr_load_matrix_market": (C.c_int, [CSR_P, C.c_char_p]),
    "spmv_b200_csr_save_matrix_market": (C.c_int, [CSR_P, C.c_char_p]),
    "spmv_b200_csr_from_coo_device": (C.c_int, [CSR_P, C.c_int, C.c_int, C.c_longlong, vp, vp, vp]),
    "spmv_b200_csr_normalize_columns_device": (C.c_int, [CSR_P]),
    "spmv_b200_csr_plan_create": (C.c_int, [CSR_P, C.c_int, C.c_int, C.POINTER(vp)]),
    "spmv_b200_csr_plan_destroy": (None, [vp]),
    "spmv_b200_csr_plan_refresh_values": (C.c_int, [vp, vp]),
    "spmv_b200_csr_plan_info": (C.c_int, [vp, c_int_p, C.POINTER(C.c_longlong), c_int_p]),
    "spmv_b200_spmv_csr_planned": (C.c_int, [vp, vp, vp, vp]),
    "spmv_b200_csr_forget_plan": (None, [CSR_P]),
    "spmv_b200_set_auto_plan": (None, [C.c_int]),
    "spmv_b200_auto_plan_enabled": (C.c_int, []),
    "spmv_b200_csr_auto_plan_info": (C.c_int, [CSR_P, c_int_p, C.POINTER(C.c_longlong)]),
    "spmv_b200_pr_plan_set_hot": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "spmv_b200_pr_plan_create": (C.c_int, [CSR_P, C.c_int, C.c_int, vp, C.POINTER(vp)]),
    "spmv_b200_pr_plan_destroy": (None, [vp]),
    "spmv_b200_pr_colsum": (C.c_int, [vp, vp, vp]),
    "spmv_b200_pr_dangling_bits": (C.c_int, [vp, C.c_int, vp, vp]),
    "spmv_b200_pr_init": (C.c_int, [C.c_int, vp, vp, vp, vp]),
    "spmv_b200_pr_step": (C.c_int, [vp, vp, vp, C.c_float, vp, vp, vp, vp]),
    "spmv_b200_pr_step_p2p": (C.c_int, [vp, vp, vp, C.c_float, vp, vp, vp, C.POINTER(vp), C.c_int, C.c_int, vp]),
    "spmv_b200_pr_step_multicast": (C.c_int, [vp, vp, vp, C.c_float, vp, vp, vp, vp, C.c_int, C.c_int, vp]),
    "spmv_b200_ipc_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp), C.c_char_p]),
    "spmv_b200_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "spmv_b200_ipc_close": (C.c_int, [vp]),
    "spmv_b200_ipc_free": (C.c_int, [vp]),
    "spmv_b200_pr_normalize": (C.c_int, [vp, C.c_int, vp, vp]),
    "spmv_b200_pagerank_device_history": (C.c_int, [CSR_P, PRC_P, vp, c_int_p, c_float_p, C.POINTER(C.c_bool), c_float_p,
                                           C.c_int]),
    "spmv_b200_pagerank_device": (C.c_int, [CSR_P, PRC_P, vp, c_int_p, c_float_p, C.POINTER(C.c_bool), c_double_p]),
    "spmv_b200_pagerank_personalized": (C.c_int, [CSR_P, PRC_P, c_float_p, PRR_P]),
    "spmv_b200_pagerank_device_personalized": (C.c_int, [CSR_P, PRC_P, c_float_p, vp, c_int_p, c_float_p,
                                                         C.POINTER(C.c_bool), c_double_p, c_float_p, C.c_int]),
    "spmv_b200_pagerank_multi_personalized": (C.c_int, [CSR_P, vp, c_float_p, C.c_int, c_int_p, C.c_int, C.c_int, C.c_int,
                                                        vp, vp]),
    "spmv_b200_pr_dist_set_personalization": (C.c_int, [vp, c_float_p]),
}


# ---- include/spmv_b200_ppr.h: the companion library libspmv_b200_ppr.so (batched personalized PageRank) ----
PPR_LIB_PATH = os.path.join(os.path.dirname(LIB_PATH), "libspmv_b200_ppr.so")

PPR_PROTOTYPES = {
    "spmv_b200_pagerank_personalized_batch": (C.c_int, [CSR_P, PRC_P, C.c_int, c_int_p, c_int_p, c_float_p, C.c_void_p,
                                                        c_int_p, c_float_p, C.POINTER(C.c_bool), c_float_p, C.c_int]),
    "spmv_b200_ppr_launch_count": (C.c_ulonglong, []),
}


def load_ppr(path=PPR_LIB_PATH):
    """dlopen libspmv_b200_ppr.so (it loads libspmv_b200.so from its own directory) and attach prototypes."""
    if not os.path.exists(path):
        raise ImportError(f"{path} not found: build it with `make -C gpu-spmv_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in PPR_PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


# ---- include/spmv_b200_ppr_topk.h: libspmv_b200_ppr_topk.so (per-seed top-K personalized PageRank) ----
PPR_TOPK_LIB_PATH = os.path.join(os.path.dirname(LIB_PATH), "libspmv_b200_ppr_topk.so")

PPR_TOPK_PROTOTYPES = {
    "spmv_b200_pagerank_personalized_batch_top_k": (C.c_int, [CSR_P, PRC_P, C.c_int, c_int_p, c_int_p, c_float_p, C.c_int,
                                                              C.c_void_p, C.c_void_p, c_int_p, c_float_p,
                                                              C.POINTER(C.c_bool), c_float_p, C.c_int]),
    "spmv_b200_ppr_topk_launch_count": (C.c_ulonglong, []),
}


def load_ppr_topk(path=PPR_TOPK_LIB_PATH):
    """dlopen libspmv_b200_ppr_topk.so (it loads libspmv_b200.so from its own directory) and attach prototypes."""
    if not os.path.exists(path):
        raise ImportError(f"{path} not found: build it with `make -C gpu-spmv_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in PPR_TOPK_PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


def load(path=LIB_PATH):
    """dlopen the library and attach prototypes.  Raises if it is missing:
    there is deliberately no fallback implementation."""
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C gpu-spmv_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    return lib
