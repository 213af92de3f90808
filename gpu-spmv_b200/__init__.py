"""gpu_spmv_b200 -- Python mirror of the LessUp/gpu-spmv API over libspmv_b200.so.

The directory is named ``gpu-spmv_b200`` (not importable by name); load it with
``_load_pkg.py`` at the repository root, which registers it as
``gpu_spmv_b200``.

Every function below has the name, argument order and error behaviour of the
reference C++ function it mirrors (include/spmv/*.h of the reference) and is a
thin ctypes call into the C ABI (include/spmv_b200.h).  Host arrays are numpy
float32/int32; device pointers are torch CUDA tensors or raw integer
addresses.  There is no CPU fallback: importing fails if the shared library
has not been built, and device calls fail if no B200 is present.
"""
import ctypes as C
import enum
import os

import numpy as np

from . import capi
from .capi import (BandwidthMetrics, BenchmarkConfig, BenchmarkResult, CSRMatrix, CSRStats, ELLMatrix,
                   PageRankConfig, PageRankResult, SpMVConfig, SpMVResult, TopKNode)

lib = capi.load()

SCALAR_CSR, VECTOR_CSR, MERGE_PATH, ELL_KERNEL = 0, 1, 2, 3
KERNEL_NAMES = {0: "SCALAR_CSR", 1: "VECTOR_CSR", 2: "MERGE_PATH", 3: "ELL_KERNEL"}


class SpMVError(enum.IntEnum):  # include/spmv/common.h:13-23
    SUCCESS = 0
    INVALID_DIMENSION = -1
    CUDA_MALLOC = -2
    CUDA_MEMCPY = -3
    KERNEL_LAUNCH = -4
    INVALID_FORMAT = -5
    FILE_IO = -6
    OUT_OF_MEMORY = -7
    INVALID_ARGUMENT = -8


def spmv_error_string(code):
    return lib.spmv_b200_error_string(int(code)).decode()


# ---------------------------------------------------------------- pointers ----

def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(capi.c_float_p)


def _i32(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(capi.c_int_p)


def dptr(t):
    """Device address of a torch CUDA tensor (or pass an int / None through)."""
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())


def host_array(ptr, n, dtype):
    """numpy view (no copy) of a host array owned by a matrix struct."""
    if not ptr or n <= 0:
        return np.empty(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(int(n),))


# --------------------------------------------------------------------- CSR ----

def csr_create(rows, cols, nnz):
    return lib.spmv_b200_csr_create(rows, cols, nnz)


def csr_destroy(mat):
    lib.spmv_b200_csr_destroy(mat)


def csr_from_dense(csr, dense, rows, cols):
    _keep, p = _f32(dense)
    return lib.spmv_b200_csr_from_dense(csr, p, rows, cols)


def csr_to_dense(csr):
    m = csr.contents
    out = np.empty(m.num_rows * m.num_cols, dtype=np.float32)
    rc = lib.spmv_b200_csr_to_dense(csr, out.ctypes.data_as(capi.c_float_p))
    return rc, out.reshape(m.num_rows, m.num_cols)


def csr_get_element(mat, row, col):
    return lib.spmv_b200_csr_get_element(mat, row, col)


def csr_to_gpu(mat):
    return lib.spmv_b200_csr_to_gpu(mat)


def csr_from_gpu(mat):
    return lib.spmv_b200_csr_from_gpu(mat)


def csr_free_gpu(mat):
    lib.spmv_b200_csr_free_gpu(mat)


def csr_serialize(mat, filename):
    return lib.spmv_b200_csr_serialize(mat, str(filename).encode())


def csr_deserialize(mat, filename):
    return lib.spmv_b200_csr_deserialize(mat, str(filename).encode())


def csr_compute_stats(mat):
    s = CSRStats()
    lib.spmv_b200_csr_compute_stats(mat, C.byref(s))
    return s


def csr_arrays(mat):
    """(row_ptrs, col_indices, values) numpy views of the host arrays."""
    m = mat.contents
    return (host_array(m.row_ptrs, m.num_rows + 1, np.int32), host_array(m.col_indices, m.nnz, np.int32),
            host_array(m.values, m.nnz, np.float32))


def csr_from_arrays(rows, cols, row_ptrs, col_indices, values):
    """csr_create + copy of caller arrays into the library-owned host arrays."""
    nnz = int(len(values))
    mat = csr_create(rows, cols, nnz)
    rp, ci, va = csr_arrays(mat)
    rp[:] = np.asarray(row_ptrs, dtype=np.int32)
    if nnz:
        ci[:] = np.asarray(col_indices, dtype=np.int32)
        va[:] = np.asarray(values, dtype=np.float32)
    return mat


class DeviceCSR:
    """Non-owning CSRMatrix over device arrays held by torch tensors (the
    struct's public d_* fields are the API's way to supply device data)."""

    def __init__(self, rows, cols, row_ptrs, col_indices, values, nnz=None):
        self._keep = (row_ptrs, col_indices, values)
        self.struct = CSRMatrix()
        self.struct.num_rows, self.struct.num_cols = int(rows), int(cols)
        self.struct.nnz = int(values.numel()) if nnz is None else int(nnz)
        self.struct.d_row_ptrs = row_ptrs.data_ptr()
        self.struct.d_col_indices = col_indices.data_ptr() if col_indices.numel() else None
        self.struct.d_values = values.data_ptr() if values.numel() else None
        self.struct.owns_host_memory = False
        self.struct.owns_device_memory = False
        self.ptr = C.pointer(self.struct)


class DeviceELL:
    """Non-owning ELLMatrix over device arrays held by torch tensors."""

    def __init__(self, rows, cols, width, col_indices, values):
        self._keep = (col_indices, values)
        self.struct = ELLMatrix()
        self.struct.num_rows, self.struct.num_cols, self.struct.max_nnz_per_row = int(rows), int(cols), int(width)
        self.struct.d_col_indices = col_indices.data_ptr() if col_indices.numel() else None
        self.struct.d_values = values.data_ptr() if values.numel() else None
        self.struct.owns_host_memory = False
        self.struct.owns_device_memory = False
        self.ptr = C.pointer(self.struct)


# --------------------------------------------------------------------- ELL ----

def ell_create(rows, cols, max_nnz_per_row):
    return lib.spmv_b200_ell_create(rows, cols, max_nnz_per_row)


def ell_destroy(mat):
    lib.spmv_b200_ell_destroy(mat)


def ell_from_dense(ell, dense, rows, cols):
    _keep, p = _f32(dense)
    return lib.spmv_b200_ell_from_dense(ell, p, rows, cols)


def ell_from_csr(ell, csr):
    return lib.spmv_b200_ell_from_csr(ell, csr)


def ell_to_dense(ell):
    m = ell.contents
    out = np.empty(m.num_rows * m.num_cols, dtype=np.float32)
    rc = lib.spmv_b200_ell_to_dense(ell, out.ctypes.data_as(capi.c_float_p))
    return rc, out.reshape(m.num_rows, m.num_cols)


def ell_get_element(mat, row, col):
    return lib.spmv_b200_ell_get_element(mat, row, col)


def ell_to_gpu(mat):
    return lib.spmv_b200_ell_to_gpu(mat)


def ell_from_gpu(mat):
    return lib.spmv_b200_ell_from_gpu(mat)


def ell_free_gpu(mat):
    lib.spmv_b200_ell_free_gpu(mat)


def ell_serialize(mat, filename):
    return lib.spmv_b200_ell_serialize(mat, str(filename).encode())


def ell_deserialize(mat, filename):
    return lib.spmv_b200_ell_deserialize(mat, str(filename).encode())


def ell_index(row, k, num_rows):
    return lib.spmv_b200_ell_index(row, k, num_rows)


def ell_arrays(mat):
    """(col_indices, values) numpy views of the host arrays (column-major)."""
    m = mat.contents
    n = m.num_rows * m.max_nnz_per_row
    return host_array(m.col_indices, n, np.int32), host_array(m.values, n, np.float32)


def ell_from_csr_device(ell, csr):
    return lib.spmv_b200_ell_from_csr_device(ell, csr)


# -------------------------------------------------------------------- SpMV ----

def make_config(kernel_type=SCALAR_CSR, block_size=256, use_texture=False):
    c = SpMVConfig()
    c.kernel_type, c.block_size, c.use_texture = int(kernel_type), int(block_size), bool(use_texture)
    return c


def spmv_cpu_csr(A, x):
    """The API's host reference function (NOT used by any device path)."""
    _keep, px = _f32(x)
    y = np.empty(A.contents.num_rows, dtype=np.float32)
    lib.spmv_b200_spmv_cpu_csr(A, px, y.ctypes.data_as(capi.c_float_p))
    return y


def spmv_cpu_ell(A, x):
    _keep, px = _f32(x)
    y = np.empty(A.contents.num_rows, dtype=np.float32)
    lib.spmv_b200_spmv_cpu_ell(A, px, y.ctypes.data_as(capi.c_float_p))
    return y


def spmv_csr(A, d_x, d_y, config=None, vec_size=-1):
    res = SpMVResult()
    cfg = C.byref(config) if config is not None else None
    lib.spmv_b200_spmv_csr(A, dptr(d_x), dptr(d_y), cfg, int(vec_size), C.byref(res))
    return res


def spmv_ell(A, d_x, d_y, config=None, vec_size=-1):
    res = SpMVResult()
    cfg = C.byref(config) if config is not None else None
    lib.spmv_b200_spmv_ell(A, dptr(d_x), dptr(d_y), cfg, int(vec_size), C.byref(res))
    return res


def spmv_csr_async(A, d_x, d_y, config=None, stream=0):
    cfg = C.byref(config) if config is not None else None
    return lib.spmv_b200_spmv_csr_async(A, dptr(d_x), dptr(d_y), cfg, C.c_void_p(stream))


def spmv_ell_async(A, d_x, d_y, stream=0):
    return lib.spmv_b200_spmv_ell_async(A, dptr(d_x), dptr(d_y), C.c_void_p(stream))


def spmv_auto_config(A):
    c = SpMVConfig()
    rc = lib.spmv_b200_auto_config(A, C.byref(c))
    if rc != 0:
        raise ValueError(spmv_error_string(rc))
    return c


def spmv_reference_policy(A):
    c = SpMVConfig()
    rc = lib.spmv_b200_reference_policy(A, C.byref(c))
    if rc != 0:
        raise ValueError(spmv_error_string(rc))
    return c


def spmv_validate_dimensions(num_cols, vec_size):
    return bool(lib.spmv_b200_validate_dimensions(num_cols, vec_size))


# --------------------------------------------------------------- bandwidth ----

def compute_bandwidth_csr(A, elapsed_ms):
    m = BandwidthMetrics()
    lib.spmv_b200_bandwidth_csr(A, float(elapsed_ms), C.byref(m))
    return m


def compute_bandwidth_ell(A, elapsed_ms):
    m = BandwidthMetrics()
    lib.spmv_b200_bandwidth_ell(A, float(elapsed_ms), C.byref(m))
    return m


def get_gpu_peak_bandwidth():
    return lib.spmv_b200_peak_bandwidth()


def csr_bytes(rows, cols, nnz):
    """Compulsory (algorithmic) bytes of one CSR SpMV, reference src/bandwidth.cpp:34-42."""
    return 8 * nnz + 4 * (rows + 1) + 4 * cols + 4 * rows


def ell_bytes(rows, cols, width):
    """Compulsory bytes of one ELL SpMV, reference src/bandwidth.cpp:66-75."""
    return 8 * rows * width + 4 * cols + 4 * rows


# ---------------------------------------------------------------- PageRank ----

def make_pagerank_config(damping_factor=0.85, tolerance=1e-6, max_iterations=100):
    c = PageRankConfig()
    c.damping_factor, c.tolerance, c.max_iterations = damping_factor, tolerance, max_iterations
    return c


def pagerank(adj_matrix, config=None):
    """Returns (PageRankResult, ranks ndarray copy); call pagerank_free(result) when done."""
    res = PageRankResult()
    cfg = C.byref(config) if config is not None else None
    rc = lib.spmv_b200_pagerank(adj_matrix, cfg, C.byref(res))
    if rc != 0:
        raise RuntimeError(f"pagerank: {spmv_error_string(rc)}")
    n = adj_matrix.contents.num_rows if adj_matrix else 0
    ranks = host_array(res.ranks, n, np.float32).copy() if res.ranks else None
    return res, ranks


def pagerank_free(result):
    lib.spmv_b200_pagerank_free(C.byref(result))


def pagerank_top_k(ranks, k):
    """Top-k of a host rank vector -> (node ids, ranks), descending."""
    ranks = np.ascontiguousarray(ranks, dtype=np.float32)
    res = PageRankResult()
    res.ranks = ranks.ctypes.data_as(capi.c_float_p)
    kk = min(k, len(ranks))
    out = (TopKNode * max(kk, 1))()
    lib.spmv_b200_pagerank_top_k(C.byref(res), len(ranks), k, out)
    return (np.array([out[i].node_id for i in range(kk)], dtype=np.int32),
            np.array([out[i].rank for i in range(kk)], dtype=np.float32))


def pagerank_top_k_device(d_ranks, k):
    """Top-k of a DEVICE rank vector (torch float32) -> (node ids, ranks), rank descending, id ascending on ties."""
    n = int(d_ranks.numel())
    kk = min(k, n)
    out = (TopKNode * max(kk, 1))()
    rc = lib.spmv_b200_pagerank_top_k_device(dptr(d_ranks), n, int(k), out)
    if rc != 0:
        raise RuntimeError(f"pagerank_top_k_device: {spmv_error_string(rc)}")
    return (np.array([out[i].node_id for i in range(kk)], dtype=np.int32),
            np.array([out[i].rank for i in range(kk)], dtype=np.float32))


def pagerank_device(adj_matrix, d_ranks, config=None):
    """Whole loop on the device; d_ranks (torch float32 [n]) receives the ranks."""
    it, res, conv, l1 = C.c_int(0), C.c_float(0), C.c_bool(False), C.c_double(0)
    cfg = C.byref(config) if config is not None else None
    rc = lib.spmv_b200_pagerank_device(adj_matrix, cfg, dptr(d_ranks), C.byref(it), C.byref(res), C.byref(conv),
                                       C.byref(l1))
    return rc, it.value, res.value, conv.value, l1.value


def pagerank_device_history(adj_matrix, d_ranks, config=None, capacity=100):
    """pagerank_device + the L2 residual of every iteration -> (rc, iterations, residual, converged, history)."""
    it, res, conv = C.c_int(0), C.c_float(0), C.c_bool(False)
    hist = np.full(capacity, np.nan, dtype=np.float32)
    cfg = C.byref(config) if config is not None else None
    rc = lib.spmv_b200_pagerank_device_history(adj_matrix, cfg, dptr(d_ranks), C.byref(it), C.byref(res), C.byref(conv),
                                               hist.ctypes.data_as(capi.c_float_p), capacity)
    return rc, it.value, res.value, conv.value, hist


def _personalization(personalization, n):
    """Host float32 copy of a personalization vector of n entries, or None."""
    if personalization is None:
        return None
    v = np.ascontiguousarray(personalization, dtype=np.float32)
    if v.ndim != 1 or v.size != n:
        raise ValueError(f"personalization must hold {n} entries, got shape {v.shape}")
    return v


def pagerank_personalized(adj_matrix, personalization, config=None):
    """Personalized PageRank: teleport and dangling mass follow `personalization` (non-negative host
    array of num_rows entries, normalised by the library; None: pagerank()).  Returns
    (PageRankResult, ranks ndarray copy); call pagerank_free(result) when done.  Raises on a rejected
    vector (NaN, Inf, negative entry, zero sum)."""
    n = adj_matrix.contents.num_rows if adj_matrix else 0
    v = _personalization(personalization, n)
    res = PageRankResult()
    cfg = C.byref(config) if config is not None else None
    rc = lib.spmv_b200_pagerank_personalized(adj_matrix, cfg, v.ctypes.data_as(capi.c_float_p) if v is not None else None,
                                             C.byref(res))
    if rc != 0:
        raise RuntimeError(f"pagerank_personalized: {spmv_error_string(rc)}")
    ranks = host_array(res.ranks, n, np.float32).copy() if res.ranks else None
    return res, ranks


def pagerank_device_personalized(adj_matrix, d_ranks, personalization, config=None, capacity=0):
    """pagerank_device for personalized PageRank (see pagerank_personalized); d_ranks (torch float32 [n])
    receives the ranks -> (rc, iterations, residual, converged, l1, history of `capacity` L2 residuals)."""
    n = adj_matrix.contents.num_rows if adj_matrix else 0
    v = _personalization(personalization, n)
    it, res, conv, l1 = C.c_int(0), C.c_float(0), C.c_bool(False), C.c_double(0)
    hist = np.full(capacity, np.nan, dtype=np.float32)
    cfg = C.byref(config) if config is not None else None
    rc = lib.spmv_b200_pagerank_device_personalized(
        adj_matrix, cfg, v.ctypes.data_as(capi.c_float_p) if v is not None else None, dptr(d_ranks), C.byref(it),
        C.byref(res), C.byref(conv), C.byref(l1), hist.ctypes.data_as(capi.c_float_p) if capacity > 0 else None, capacity)
    return rc, it.value, res.value, conv.value, l1.value, hist


# ------------------------------------------- batched personalized PageRank (libspmv_b200_ppr.so) ----
_ppr = None


def ppr_lib():
    """libspmv_b200_ppr.so, loaded on first use: importing the package does not need the companion."""
    global _ppr
    if _ppr is None:
        _ppr = capi.load_ppr()
    return _ppr


def _teleport_columns(V, n):
    """(k, offsets, nodes, weights) of the sparse column form of V; weights None means all 1."""
    try:
        import scipy.sparse as S
        if S.issparse(V):
            M = S.csr_matrix(V)
            if M.ndim != 2 or M.shape[1] != n:
                raise ValueError(f"a sparse V must be (k, {n}), got {M.shape}")
            M = M.sorted_indices()
            return (M.shape[0], np.ascontiguousarray(M.indptr, np.int32), np.ascontiguousarray(M.indices, np.int32),
                    np.ascontiguousarray(M.data, np.float32))
    except ImportError:
        pass
    V = np.asarray(V)
    if V.ndim == 1:  # seed node ids: one-hot vectors
        if V.size and not np.issubdtype(V.dtype, np.integer):
            raise ValueError("a 1-D V holds seed node ids (integers)")
        k = V.size
        return k, np.arange(k + 1, dtype=np.int32), np.ascontiguousarray(V, np.int32), None
    if V.ndim != 2 or V.shape[1] != n:
        raise ValueError(f"a dense V must be (k, {n}), got shape {V.shape}")
    V = np.ascontiguousarray(V, np.float32)
    rows, cols = np.nonzero(V)  # row-major order: ascending nodes per column; zeros add nothing to the sum
    offsets = np.zeros(V.shape[0] + 1, np.int32)
    offsets[1:] = np.cumsum(np.bincount(rows, minlength=V.shape[0]))
    return V.shape[0], offsets, cols.astype(np.int32), V[rows, cols]


def pagerank_personalized_batch(A, V, config=None, capacity=0):
    """k personalized PageRank vectors of the graph A (device CSR) in one loop.

    V: a 1-D sequence of seed node ids (one-hot teleport vectors), a dense (k, n) array, or a scipy.sparse (k, n)
    matrix; each row is normalised by the library, as in pagerank_personalized.  Returns (ranks, iterations,
    residual, converged, history): ranks is an (n, k) float32 torch tensor on the current CUDA device (column c is
    vector c), the others are per-column numpy arrays; history is (k, capacity), NaN beyond a column's iterations.
    Raises RuntimeError with the library's status on a rejected input."""
    import torch
    lib_p = ppr_lib()
    n = A.contents.num_rows if A else 0
    k, offsets, nodes, weights = _teleport_columns(V, n)
    ranks = torch.empty((n, k), dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
    it = np.zeros(k, np.int32)
    res = np.zeros(k, np.float32)
    conv = np.zeros(k, np.bool_)
    hist = np.full((k, capacity), np.nan, dtype=np.float32)
    cfg = C.byref(config) if config is not None else None
    rc = lib_p.spmv_b200_pagerank_personalized_batch(
        A, cfg, k, offsets.ctypes.data_as(capi.c_int_p), nodes.ctypes.data_as(capi.c_int_p),
        weights.ctypes.data_as(capi.c_float_p) if weights is not None else None, dptr(ranks), it.ctypes.data_as(capi.c_int_p),
        res.ctypes.data_as(capi.c_float_p), conv.ctypes.data_as(C.POINTER(C.c_bool)),
        hist.ctypes.data_as(capi.c_float_p) if capacity > 0 else None, capacity)
    if rc != 0:
        raise RuntimeError(f"pagerank_personalized_batch: {spmv_error_string(rc)}")
    return ranks, it, res, conv, hist


# ------------------------------- per-seed top-K personalized PageRank (libspmv_b200_ppr_topk.so) ----
_ppr_topk = None


def ppr_topk_lib():
    """libspmv_b200_ppr_topk.so, loaded on first use: importing the package does not need it."""
    global _ppr_topk
    if _ppr_topk is None:
        _ppr_topk = capi.load_ppr_topk()
    return _ppr_topk


def pagerank_personalized_batch_top_k(A, V, top, config=None, capacity=0):
    """The `top` best nodes of each of k personalized PageRank vectors of the graph A (device CSR), without the
    dense (n, k) rank matrix.

    V as in pagerank_personalized_batch.  Returns (ids, vals, iterations, residual, converged, history): ids (int32)
    and vals (float32) are (k, top) torch tensors on the current CUDA device; row c holds the min(top, n) largest
    ranks of vector c, bit for bit those of pagerank_personalized_batch, by rank descending then node id ascending,
    padded with (-1, 0.0).  The others are as in pagerank_personalized_batch.  Raises RuntimeError with the
    library's status on a rejected input (top outside [1, 1024] among them)."""
    import torch
    lib_t = ppr_topk_lib()
    n = A.contents.num_rows if A else 0
    k, offsets, nodes, weights = _teleport_columns(V, n)
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = max(int(top), 0)
    ids = torch.empty((k, rows), dtype=torch.int32, device=dev)
    vals = torch.empty((k, rows), dtype=torch.float32, device=dev)
    it = np.zeros(k, np.int32)
    res = np.zeros(k, np.float32)
    conv = np.zeros(k, np.bool_)
    hist = np.full((k, capacity), np.nan, dtype=np.float32)
    cfg = C.byref(config) if config is not None else None
    rc = lib_t.spmv_b200_pagerank_personalized_batch_top_k(
        A, cfg, k, offsets.ctypes.data_as(capi.c_int_p), nodes.ctypes.data_as(capi.c_int_p),
        weights.ctypes.data_as(capi.c_float_p) if weights is not None else None, int(top), dptr(ids), dptr(vals),
        it.ctypes.data_as(capi.c_int_p), res.ctypes.data_as(capi.c_float_p), conv.ctypes.data_as(C.POINTER(C.c_bool)),
        hist.ctypes.data_as(capi.c_float_p) if capacity > 0 else None, capacity)
    if rc != 0:
        raise RuntimeError(f"pagerank_personalized_batch_top_k: {spmv_error_string(rc)}")
    return ids, vals, it, res, conv, hist


# --------------------------------------------------------------- benchmark ----

def make_bench_config(num_warmup_runs=5, num_runs=20, compare_cpu=True):
    c = BenchmarkConfig()
    c.num_warmup_runs, c.num_runs, c.compare_cpu = num_warmup_runs, num_runs, compare_cpu
    return c


def benchmark_csr(A, x, config=None, bench_config=None):
    _keep, px = _f32(x)
    out = BenchmarkResult()
    rc = lib.spmv_b200_benchmark_csr(A, px, C.byref(config) if config is not None else None,
                                     C.byref(bench_config) if bench_config is not None else None, C.byref(out))
    if rc != 0:
        raise RuntimeError(f"benchmark_csr: {spmv_error_string(rc)}")
    return out


def benchmark_ell(A, x, bench_config=None):
    _keep, px = _f32(x)
    out = BenchmarkResult()
    rc = lib.spmv_b200_benchmark_ell(A, px, C.byref(bench_config) if bench_config is not None else None, C.byref(out))
    if rc != 0:
        raise RuntimeError(f"benchmark_ell: {spmv_error_string(rc)}")
    return out


def compare_gpu_cpu_csr(A, x, config=None, bench_config=None):
    _keep, px = _f32(x)
    gpu, cpu, speedup = BenchmarkResult(), BenchmarkResult(), C.c_float(0)
    rc = lib.spmv_b200_compare_gpu_cpu_csr(A, px, C.byref(config) if config is not None else None,
                                           C.byref(bench_config) if bench_config is not None else None,
                                           C.byref(gpu), C.byref(cpu), C.byref(speedup))
    if rc != 0:
        raise RuntimeError(f"compare_gpu_cpu_csr: {spmv_error_string(rc)}")
    return gpu, cpu, speedup.value


def benchmark_to_json(result):
    buf = C.create_string_buffer(4096)
    n = lib.spmv_b200_benchmark_to_json(C.byref(result), buf, 4096)
    if n < 0:
        raise RuntimeError("benchmark_to_json failed")
    return buf.value.decode()


def benchmark_from_json(text):
    out = BenchmarkResult()
    lib.spmv_b200_benchmark_from_json(text.encode(), C.byref(out))
    return out


# -------------------------------------------------------------- extensions ----

def launch_count():
    return int(lib.spmv_b200_launch_count())


def csr_load_matrix_market(mat, filename):
    return lib.spmv_b200_csr_load_matrix_market(mat, os.fsencode(filename))


def csr_save_matrix_market(mat, filename):
    return lib.spmv_b200_csr_save_matrix_market(mat, os.fsencode(filename))


def csr_from_coo_device(out, rows, cols, d_rows, d_cols, d_vals):
    """Device COO (torch int32 / int32 / float32 tensors) -> device CSR in `out` (a csr_create handle)."""
    return lib.spmv_b200_csr_from_coo_device(out, int(rows), int(cols), int(d_vals.numel()), dptr(d_rows), dptr(d_cols),
                                             dptr(d_vals))


def csr_normalize_columns_device(A):
    return lib.spmv_b200_csr_normalize_columns_device(A)


class CsrPlan:
    """Merge coordinates + hub-column table of a device CSR (spmv_b200_csr_plan)."""

    def __init__(self, A, max_hot_columns=0, force=False, snapshot_values=False):
        self.handle = C.c_void_p()
        flags = (1 if force else 0) | (2 if snapshot_values else 0)
        rc = lib.spmv_b200_csr_plan_create(A, int(max_hot_columns), flags, C.byref(self.handle))
        if rc != 0:
            raise RuntimeError(f"csr_plan_create: {spmv_error_string(rc)}")
        self._A = A  # the plan reads the matrix's device arrays

    def info(self):
        """(hot_columns, hot_nnz, mode); mode 0 plain tile kernel, 1 / 2 hub-column kernel (table / all of x),
        3 / 4 segmented stream, 5 ELL layout (snapshot of the values)."""
        n, z, m = C.c_int(0), C.c_longlong(0), C.c_int(0)
        lib.spmv_b200_csr_plan_info(self.handle, C.byref(n), C.byref(z), C.byref(m))
        return n.value, z.value, m.value

    def spmv(self, d_x, d_y, stream=0):
        return lib.spmv_b200_spmv_csr_planned(self.handle, dptr(d_x), dptr(d_y), C.c_void_p(stream))

    def refresh_values(self, stream=0):
        """Re-reads d_values into the ELL snapshot of a mode-5 plan (no-op otherwise)."""
        return lib.spmv_b200_csr_plan_refresh_values(self.handle, C.c_void_p(stream))

    def close(self):
        if self.handle:
            lib.spmv_b200_csr_plan_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def csr_forget_plan(A):
    lib.spmv_b200_csr_forget_plan(A)


def csr_auto_plan_info(A):
    """(hot_columns, hot_nnz) of the plan spmv_csr(MERGE_PATH) attached to A's upload, (0, 0) if none."""
    n, z = C.c_int(0), C.c_longlong(0)
    lib.spmv_b200_csr_auto_plan_info(A, C.byref(n), C.byref(z))
    return n.value, z.value


def merge_path_search(diagonal, row_ptrs, num_rows, nnz):
    _keep, p = _i32(row_ptrs)
    r, z = C.c_int(0), C.c_int(0)
    rc = lib.spmv_b200_merge_path_search(diagonal, p, num_rows, nnz, C.byref(r), C.byref(z))
    if rc != 0:
        raise ValueError(spmv_error_string(rc))
    return r.value, z.value


def partition_rows(row_ptrs, num_rows, parts, row_weight=0):
    """Contiguous row split balancing nnz(row) + row_weight (0: nnz-balanced, 1: merge items)."""
    _keep, p = _i32(row_ptrs)
    bounds = np.zeros(parts + 1, dtype=np.int32)
    rc = lib.spmv_b200_partition_rows_weighted(p, num_rows, parts, int(row_weight), bounds.ctypes.data_as(capi.c_int_p))
    if rc != 0:
        raise ValueError(spmv_error_string(rc))
    return bounds
