"""Row-sharded SpMV / PageRank for one process per GPU.

The reference has no multi-GPU code (SURVEY 2, 8e); this is the additive extension BASELINE.json asks
for.  Rows are split into contiguous work-balanced shards (`partition_rows`, the rule of
spmv_b200_partition_rows_weighted), and `extract_shard` cuts one out as a stand-alone CSR that keeps
global column ids, so every rank holds a full-length rank vector.

`CudaShard` is a thin ctypes face of the per-shard building blocks of include/spmv_b200.h (plan,
column sums, dangling bits, start vector, fused step, normalisation), for callers that write their own
loop.  The sharded PageRank itself is native (csrc/pagerank_dist.cu): `NativeComm` and
`NativeShardedPageRank` only pass pointers to it, and the library does the rendezvous, symmetric
buffers, slice exchange, stop rule and CUDA-graph replay.
"""
import ctypes as C

import numpy as np
import torch

import gpu_spmv_b200 as sp
import gpu_spmv_b200.gen as gen


# ------------------------------------------------------------- partitioning ----

def partition_rows(row_ptrs, parts, row_weight=0):
    """Contiguous row split balancing work(row) = nnz(row) + row_weight (0: nnz-balanced; 1: the
    merge-path items rows + nnz that the merge-path / PageRank kernels consume).  row_ptrs is a
    host int32 array or a torch tensor (any device).  Returns a list of parts+1 row bounds."""
    if torch.is_tensor(row_ptrs) and row_ptrs.is_cuda:
        return gen.partition_bounds(row_ptrs, parts, row_weight)
    rp = np.ascontiguousarray(row_ptrs.numpy() if torch.is_tensor(row_ptrs) else row_ptrs, dtype=np.int32)
    return [int(b) for b in sp.partition_rows(rp, len(rp) - 1, parts, row_weight)]


def extract_shard(row_ptrs, col_indices, values, lo, hi):
    """Rows [lo, hi) as a stand-alone CSR: row_ptrs rebased to 0, global column ids."""
    a, b = int(row_ptrs[lo]), int(row_ptrs[hi])
    rp = (row_ptrs[lo:hi + 1] - row_ptrs[lo]).contiguous()
    return rp, col_indices[a:b].contiguous(), values[a:b].contiguous()


# ------------------------------------------------------ per-shard building blocks ----

class CudaShard:
    """This rank's row shard on its GPU plus the fused-iteration plan."""

    def __init__(self, n_global, row_lo, row_ptrs, col_indices, values, stream=None):
        self.n = int(n_global)
        self.row_lo = int(row_lo)
        self.rows = row_ptrs.numel() - 1
        self.dev = row_ptrs.device
        self.csr = sp.DeviceCSR(self.rows, self.n, row_ptrs, col_indices, values)
        self.stream = stream
        handle = C.c_void_p()
        rc = sp.lib.spmv_b200_pr_plan_create(self.csr.ptr, self.row_lo, self.n, self._s(), C.byref(handle))
        if rc != 0:
            raise RuntimeError(f"pr_plan_create: {sp.spmv_error_string(rc)}")
        self.plan = handle
        self.bits = torch.zeros((self.n + 31) // 32, dtype=torch.int32, device=self.dev)
        self.dsum = torch.zeros(1, dtype=torch.float32, device=self.dev)
        self.damping = 0.85

    def _s(self):
        return C.c_void_p(self.stream if self.stream is not None else torch.cuda.current_stream().cuda_stream)

    def close(self):
        if self.plan:
            sp.lib.spmv_b200_pr_plan_destroy(self.plan)
            self.plan = None

    def set_hot(self, max_hot_columns=-1, force=False):
        """Rebuilds the shard's hub-column table (csr_hot_kernels.cu): 0 = none, < 0 = device
        maximum.  Returns the number of hub columns in use."""
        n = sp.lib.spmv_b200_pr_plan_set_hot(self.plan, int(max_hot_columns), int(bool(force)), self._s())
        if n < 0:
            raise RuntimeError(f"pr_plan_set_hot: {sp.spmv_error_string(n)}")
        return n

    def setup_dangling(self):
        """Dangling columns = column sums equal to 0 (src/pagerank.cu:20-48), from THIS shard's column
        sums: exact for a shard that holds the whole graph.  Over several shards, sum
        spmv_b200_pr_colsum of every shard first and build the bits from the total."""
        colsum = torch.zeros(self.n, dtype=torch.float64, device=self.dev)
        rc = sp.lib.spmv_b200_pr_colsum(self.plan, sp.dptr(colsum), self._s())
        assert rc == 0
        rc = sp.lib.spmv_b200_pr_dangling_bits(sp.dptr(colsum), self.n, sp.dptr(self.bits), self._s())
        assert rc == 0

    def init_vector(self, r):
        rc = sp.lib.spmv_b200_pr_init(self.n, sp.dptr(self.bits), sp.dptr(r), sp.dptr(self.dsum), self._s())
        assert rc == 0

    def __call__(self, r_old, r_new, partial):
        """One fused step (spmv_b200_pr_step): this shard's rows of r_new and its three partial sums
        (float64 [3]: sum d^2, sum |d|, next dangling mass), with self.dsum as r_old's dangling mass."""
        rc = sp.lib.spmv_b200_pr_step(self.plan, sp.dptr(r_old), sp.dptr(r_new), self.damping, sp.dptr(self.dsum),
                                      sp.dptr(self.bits), sp.dptr(partial), self._s())
        if rc != 0:
            raise RuntimeError(f"pr_step: {sp.spmv_error_string(rc)}")

    def normalize(self, r):
        out = torch.empty_like(r)
        rc = sp.lib.spmv_b200_pr_normalize(sp.dptr(r), self.n, sp.dptr(out), self._s())
        assert rc == 0
        return out


# ------------------------------------------- native sharded PageRank (csrc/pagerank_dist.cu) ----
# Rendezvous, symmetric memory, multicast binding, in-kernel flag barrier and CUDA-graph replay all
# live in libspmv_b200.so; Python only passes pointers.

class _RawDeviceArray:
    """float32 device memory owned by libspmv_b200 (cudaMalloc), exposed to torch without a copy."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


def _tensor_from_ptr(ptr, n, device):
    return torch.as_tensor(_RawDeviceArray(ptr, n), device=device)


EXCHANGE_AUTO, EXCHANGE_NCCL, EXCHANGE_P2P, EXCHANGE_MULTICAST = -1, 0, 1, 2
EXCHANGE_NAMES = {0: "nccl", 1: "p2p", 2: "multicast"}


class PrDistResult(C.Structure):  # include/spmv_b200.h: spmv_b200_pr_dist_result
    _fields_ = [("iterations", C.c_int), ("final_residual", C.c_float), ("converged", C.c_int),
                ("l1_residual", C.c_double), ("iterations_launched", C.c_int), ("device_seconds", C.c_double),
                ("wall_seconds", C.c_double), ("exchange", C.c_int), ("graph_replay", C.c_int),
                ("kernels_per_iteration", C.c_int)]


class NativeComm:
    """spmv_b200_comm_*: one process per GPU, abstract unix socket named after `session`."""

    def __init__(self, rank, world, session, timeout_s=300):
        self.rank, self.world = int(rank), int(world)
        self.handle = C.c_void_p()
        rc = sp.lib.spmv_b200_comm_create(self.rank, self.world, str(session).encode(), int(timeout_s), C.byref(self.handle))
        if rc != 0:
            raise RuntimeError(f"comm_create(rank {rank} of {world}, session {session}): {sp.spmv_error_string(rc)}")

    def barrier(self):
        assert sp.lib.spmv_b200_comm_barrier(self.handle) == 0

    def allgather_doubles(self, value):
        send = (C.c_double * 1)(float(value))
        recv = (C.c_double * self.world)()
        assert sp.lib.spmv_b200_comm_allgather(self.handle, send, recv, 8) == 0
        return list(recv)

    def close(self):
        if self.handle:
            sp.lib.spmv_b200_comm_destroy(self.handle)
            self.handle = None


class NativeShardedPageRank:
    """spmv_b200_pr_dist_*: this rank's shard (a DeviceCSR with global column ids) of a sharded PageRank.
    personalization: the FULL personalization vector (n_global non-negative entries, the same on every
    rank) for personalized PageRank, or None for global PageRank; set_personalization changes it later."""

    def __init__(self, comm, csr, row_offset, n_global, exchange=EXCHANGE_AUTO, personalization=None):
        self.comm, self.csr, self.n = comm, csr, int(n_global)
        self.handle = C.c_void_p()
        rc = sp.lib.spmv_b200_pr_dist_create(comm.handle, csr.ptr, int(row_offset), self.n, int(exchange), C.byref(self.handle))
        if rc != 0:
            raise RuntimeError(f"pr_dist_create: {sp.spmv_error_string(rc)}")
        self.exchange = sp.lib.spmv_b200_pr_dist_exchange(self.handle)
        self.hub_columns = sp.lib.spmv_b200_pr_dist_hub_columns(self.handle)
        if personalization is not None:
            try:
                self.set_personalization(personalization)
            except Exception:
                self.close()
                raise

    def set_personalization(self, personalization):
        """Collective: personalized PageRank from the next run on (None: global PageRank again)."""
        v = sp._personalization(personalization, self.n)
        rc = sp.lib.spmv_b200_pr_dist_set_personalization(self.handle, v.ctypes.data_as(sp.capi.c_float_p)
                                                          if v is not None else None)
        if rc != 0:
            raise RuntimeError(f"pr_dist_set_personalization: {sp.spmv_error_string(rc)}")

    def run(self, damping=0.85, tolerance=1e-6, max_iterations=100, fixed_iterations=0):
        cfg = sp.make_pagerank_config(damping, tolerance, max_iterations)
        res = PrDistResult()
        rc = sp.lib.spmv_b200_pr_dist_run(self.handle, C.byref(cfg), int(fixed_iterations), C.byref(res))
        if rc != 0:
            raise RuntimeError(f"pr_dist_run: {sp.spmv_error_string(rc)}")
        return res

    def ranks(self, device):
        ptr = sp.lib.spmv_b200_pr_dist_ranks(self.handle)
        return _tensor_from_ptr(ptr, self.n, device)

    def close(self):
        if self.handle:
            sp.lib.spmv_b200_pr_dist_destroy(self.handle)
            self.handle = None
