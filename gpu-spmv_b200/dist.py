"""Row-sharded SpMV / PageRank for one process per GPU.

The reference has no multi-GPU code (SURVEY 2, 8e); this is the additive
extension BASELINE.json asks for: rows are split into contiguous nnz-balanced
shards (spmv_b200_partition_rows), every rank keeps global column ids and a
full-length rank vector, and one PageRank iteration is

    local fused step (spmv_b200_pr_step: SpMV + damping/teleport + dangling +
                      residual partial sums, one pass over the shard)
    all-gather of the freshly written rank slices        (NCCL over NVLink)
    all-reduce of {sum d^2, sum |d|, next dangling mass} (3 doubles)

torch.distributed is plumbing only (rendezvous, NCCL communicator, streams);
the arithmetic is in libspmv_b200.so.  The loop itself (`pagerank_loop`) is
backend-agnostic so that the host logic -- partitioning, slice exchange,
reduction of the partial sums, stop rule -- is covered by world_size-2 gloo
tests on CPU with a checker-supplied local step.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

import gpu_spmv_b200 as sp


# ------------------------------------------------------------- partitioning ----

def partition_rows(row_ptrs, parts, row_weight=0):
    """Contiguous row split balancing work(row) = nnz(row) + row_weight (0: nnz-balanced; 1: the
    merge-path items rows + nnz that the merge-path / PageRank kernels consume).  row_ptrs is a
    host int32 array or a torch tensor (any device).  Returns a list of parts+1 row bounds."""
    if torch.is_tensor(row_ptrs) and row_ptrs.is_cuda:
        rows = row_ptrs.numel() - 1
        prefix = row_ptrs[:rows].to(torch.int64) + torch.arange(rows, dtype=torch.int64, device=row_ptrs.device) * row_weight
        total = int(row_ptrs[-1].item()) + rows * row_weight
        targets = torch.tensor([(total * p) // parts for p in range(1, parts)], dtype=torch.int64, device=row_ptrs.device)
        inner = torch.searchsorted(prefix, targets, right=False).tolist() if parts > 1 else []
        bounds = [0] + [int(b) for b in inner] + [rows]
        for p in range(1, parts + 1):
            bounds[p] = max(bounds[p], bounds[p - 1])
        return bounds
    rp = np.ascontiguousarray(row_ptrs.numpy() if torch.is_tensor(row_ptrs) else row_ptrs, dtype=np.int32)
    return [int(b) for b in sp.partition_rows(rp, len(rp) - 1, parts, row_weight)]


def extract_shard(row_ptrs, col_indices, values, lo, hi):
    """Rows [lo, hi) as a stand-alone CSR: row_ptrs rebased to 0, global column ids."""
    a, b = int(row_ptrs[lo]), int(row_ptrs[hi])
    rp = (row_ptrs[lo:hi + 1] - row_ptrs[lo]).contiguous()
    return rp, col_indices[a:b].contiguous(), values[a:b].contiguous()


# ------------------------------------------------------------ slice exchange ----

def all_gather_slices(full, bounds, group=None):
    """In-place all-gather of variable-length slices: on return every rank holds
    full[bounds[p]:bounds[p+1]] as written by rank p."""
    if not dist.is_initialized():
        return
    world = dist.get_world_size(group)
    if world == 1:
        return
    rank = dist.get_rank(group)
    sizes = [bounds[p + 1] - bounds[p] for p in range(world)]
    if len(set(sizes)) == 1 and sizes[0] > 0:
        dist.all_gather_into_tensor(full[bounds[0]:bounds[world]], full[bounds[rank]:bounds[rank + 1]], group=group)
        return
    views = [full[bounds[p]:bounds[p + 1]] for p in range(world)]
    if dist.get_backend(group) == "nccl" and all(s > 0 for s in sizes):
        # uneven sizes: ProcessGroupNCCL runs this as one coalesced group of broadcasts
        dist.all_gather(views, views[rank].clone(), group=group)
        return
    for p in range(world):
        if sizes[p] > 0:
            dist.broadcast(views[p], src=dist.get_global_rank(group, p) if group is not None else p, group=group)


# ----------------------------------------------------------------- the loop ----

class PageRankOutcome:
    def __init__(self, ranks, iterations, final_residual, converged, l1_residual, seconds_per_iteration=None):
        self.ranks, self.iterations, self.final_residual = ranks, iterations, final_residual
        self.converged, self.l1_residual = converged, l1_residual
        self.seconds_per_iteration = seconds_per_iteration


def pagerank_loop(step, r_old, r_new, partial, bounds, damping, tolerance, max_iterations, group=None,
                  fixed_iterations=0, on_iteration=None):
    """The reference's iteration control (src/pagerank.cu:93-139) around a sharded step.

    step(r_old, r_new, partial) must write this rank's slice of r_new and its
    three partial sums (float64 tensor [3]: sum d^2, sum |d|, next dangling mass)
    and is told the all-reduced dangling mass through step.set_dangling_mass().

    The stop rule is the reference's (L2 norm of the delta < tolerance, evaluated for EVERY
    iteration), but it is evaluated one iteration late: the 24-byte sums of iteration i are
    copied to pinned host memory asynchronously and read while iteration i+1 is already queued,
    so the device never idles on the host.  If iteration i turns out to have converged, its
    output -- the INPUT buffer of the speculative iteration i+1, which that iteration does not
    write -- is returned; iteration count, residual and vector are exactly those of the eager
    rule.  Returns (final vector, iterations, residual, converged, l1)."""
    limit = fixed_iterations if fixed_iterations > 0 else max_iterations
    on_gpu = partial.is_cuda
    host_bufs = [torch.empty(3, dtype=torch.float64, pin_memory=on_gpu) for _ in range(2)]
    events = [torch.cuda.Event() for _ in range(2)] if on_gpu else [None, None]
    distributed = dist.is_initialized() and dist.get_world_size(group) > 1

    def read(slot):
        if on_gpu:
            events[slot].synchronize()
        host = host_bufs[slot]
        res = float(np.sqrt(np.float32(host[0].item())))  # L2 norm of the delta in fp32 (src/pagerank.cu:118)
        return res, float(host[1].item())

    iters, residual, l1, conv = 0, 0.0, 0.0, False
    final = r_old       # what the reference returns when the loop never runs
    pending = None      # (iteration number, host slot, vector that iteration produced)
    for it in range(limit):
        step(r_old, r_new, partial)
        if not getattr(step, "delivers_slices", False):
            all_gather_slices(r_new, bounds, group)
        if distributed:  # with a fused exchange this all-reduce is also the barrier that orders the peer stores
            dist.all_reduce(partial, op=dist.ReduceOp.SUM, group=group)
        step.set_dangling_mass(partial)
        slot = it % 2
        host_bufs[slot].copy_(partial, non_blocking=True)
        if on_gpu:
            events[slot].record()
        if pending is not None:
            p_iter, p_slot, p_vec = pending
            residual, l1 = read(p_slot)
            iters, final = p_iter, p_vec
            if on_iteration is not None:
                on_iteration(iters, residual)
            if fixed_iterations <= 0 and residual < tolerance:
                conv = True
                pending = None
                break
        pending = (it + 1, slot, r_new)
        r_old, r_new = r_new, r_old
    if pending is not None:  # the last queued iteration
        p_iter, p_slot, p_vec = pending
        residual, l1 = read(p_slot)
        iters, final = p_iter, p_vec
        if on_iteration is not None:
            on_iteration(iters, residual)
        conv = residual < tolerance
    return final, iters, residual, conv, l1


# ------------------------------------------------------- CUDA step (product) ----

class _RawDeviceArray:
    """float32 device memory owned by libspmv_b200 (cudaMalloc), exposed to torch without a copy."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


def _tensor_from_ptr(ptr, n, device):
    return torch.as_tensor(_RawDeviceArray(ptr, n), device=device)


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
        self._peer_tables, self._world, self._rank = {}, 1, 0
        self._multicast, self._symm = {}, []

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

    def setup_dangling(self, group=None):
        """Dangling columns = global column sums equal to 0 (src/pagerank.cu:20-48)."""
        colsum = torch.zeros(self.n, dtype=torch.float64, device=self.dev)
        rc = sp.lib.spmv_b200_pr_colsum(self.plan, sp.dptr(colsum), self._s())
        assert rc == 0
        if dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(colsum, op=dist.ReduceOp.SUM, group=group)
        rc = sp.lib.spmv_b200_pr_dangling_bits(sp.dptr(colsum), self.n, sp.dptr(self.bits), self._s())
        assert rc == 0

    def init_vector(self, r):
        rc = sp.lib.spmv_b200_pr_init(self.n, sp.dptr(self.bits), sp.dptr(r), sp.dptr(self.dsum), self._s())
        assert rc == 0

    def __call__(self, r_old, r_new, partial):
        mc = self._multicast.get(r_new.data_ptr()) if self._multicast else None
        if mc is not None:  # slice exchange fused into the step, one NVSwitch-multicast store per value
            rc = sp.lib.spmv_b200_pr_step_multicast(self.plan, sp.dptr(r_old), sp.dptr(r_new), self.damping,
                                                    sp.dptr(self.dsum), sp.dptr(self.bits), sp.dptr(partial),
                                                    C.c_void_p(mc), self._world, self._rank, self._s())
            if rc != 0:
                raise RuntimeError(f"pr_step_multicast: {sp.spmv_error_string(rc)}")
            return
        table = self._peer_tables.get(r_new.data_ptr()) if self._peer_tables else None
        if table is not None:  # slice exchange fused into the step (peer stores over NVLink)
            rc = sp.lib.spmv_b200_pr_step_p2p(self.plan, sp.dptr(r_old), sp.dptr(r_new), self.damping,
                                              sp.dptr(self.dsum), sp.dptr(self.bits), sp.dptr(partial), table,
                                              self._world, self._rank, self._s())
        else:
            rc = sp.lib.spmv_b200_pr_step(self.plan, sp.dptr(r_old), sp.dptr(r_new), self.damping, sp.dptr(self.dsum),
                                          sp.dptr(self.bits), sp.dptr(partial), self._s())
        if rc != 0:
            raise RuntimeError(f"pr_step: {sp.spmv_error_string(rc)}")

    # ---- fused slice exchange: peer-mapped rank-vector buffers ---------------------------------
    @property
    def delivers_slices(self):
        """True when the step itself writes this rank's slice into every peer's vector."""
        return bool(self._peer_tables) or bool(self._multicast)

    def enable_multicast_exchange(self, group=None):
        """The two rank-vector buffers as torch symmetric memory bound to an NVSwitch multicast
        object: the step then sends every finished value ONCE (multimem.st) and the switch delivers
        it to all GPUs.  torch.distributed._symmetric_memory does the plumbing (cuMem allocation,
        handle exchange, cuMulticast* binding); returns (r_a, r_b) or None when the box / torch
        build has no multicast support (callers then fall back to enable_peer_exchange)."""
        try:
            import torch.distributed._symmetric_memory as symm_mem
            self._world, self._rank = dist.get_world_size(group), dist.get_rank(group)
            pg = group if group is not None else dist.group.WORLD
            bufs, handles = [], []
            for _ in range(2):
                t = symm_mem.empty(self.n, dtype=torch.float32, device=self.dev)
                h = symm_mem.rendezvous(t, pg)
                if not getattr(h, "multicast_ptr", 0):
                    return None
                bufs.append(t)
                handles.append(h)
        except Exception as exc:  # no symmetric memory in this build / on this box
            self._multicast_error = repr(exc)
            return None
        self._symm = handles  # keep the mappings alive
        self._multicast = {t.data_ptr(): int(h.multicast_ptr) for t, h in zip(bufs, handles)}
        return tuple(bufs)

    def disable_multicast_exchange(self):
        self._multicast, self._symm = {}, []

    def enable_peer_exchange(self, group=None):
        """Allocates the two rank-vector buffers of the iteration as CUDA-IPC shareable memory,
        maps every peer's pair into this process and returns them as torch tensors (r_a, r_b).
        Needs one process per GPU on one NVLink/NVSwitch box."""
        self._world, self._rank = dist.get_world_size(group), dist.get_rank(group)
        if self._world > 8:
            raise ValueError("peer exchange is for the <= 8 GPUs of one box")
        nbytes = self.n * 4
        mine, handles = [], []
        for _ in range(2):
            ptr, h = C.c_void_p(), C.create_string_buffer(64)
            rc = sp.lib.spmv_b200_ipc_alloc(nbytes, C.byref(ptr), h)
            if rc != 0:
                raise RuntimeError(f"ipc_alloc: {sp.spmv_error_string(rc)}")
            mine.append(ptr.value)
            handles.append(h.raw)
        everyone = [None] * self._world
        dist.all_gather_object(everyone, handles, group=group)
        self._ipc_mine, self._ipc_opened, self._peer_tables = mine, [], {}
        for b in range(2):
            table = (C.c_void_p * 8)()
            for p in range(self._world):
                if p == self._rank:
                    table[p] = mine[b]
                else:
                    ptr = C.c_void_p()
                    rc = sp.lib.spmv_b200_ipc_open(everyone[p][b], C.byref(ptr))
                    if rc != 0:
                        raise RuntimeError(f"ipc_open (rank {p}): {sp.spmv_error_string(rc)}")
                    table[p] = ptr.value
                    self._ipc_opened.append(ptr.value)
            self._peer_tables[mine[b]] = table
        return tuple(_tensor_from_ptr(ptr, self.n, self.dev) for ptr in mine)

    def disable_peer_exchange(self):
        for ptr in getattr(self, "_ipc_opened", []):
            sp.lib.spmv_b200_ipc_close(C.c_void_p(ptr))
        for ptr in getattr(self, "_ipc_mine", []):
            sp.lib.spmv_b200_ipc_free(C.c_void_p(ptr))
        self._ipc_opened, self._ipc_mine, self._peer_tables = [], [], {}

    def set_dangling_mass(self, partial):
        self.dsum.copy_(partial[2:3].to(torch.float32))

    def normalize(self, r):
        out = torch.empty_like(r)
        rc = sp.lib.spmv_b200_pr_normalize(sp.dptr(r), self.n, sp.dptr(out), self._s())
        assert rc == 0
        return out

    def spmv(self, x, y_full, kernel=sp.MERGE_PATH):
        """y_full[row_lo : row_lo + rows] = A_shard x (no collective: x is replicated)."""
        y = y_full[self.row_lo:self.row_lo + self.rows]
        return sp.spmv_csr_async(self.csr.ptr, x, y, sp.make_config(kernel), self._s().value or 0)


def pagerank_sharded(shard, bounds, damping=0.85, tolerance=1e-6, max_iterations=100, group=None,
                     fixed_iterations=0, fused_exchange=False):
    """PageRank over row shards, one CudaShard per rank; returns a PageRankOutcome whose
    ranks tensor (full length, normalised) is identical on every rank.  fused_exchange=True
    replaces the NCCL all-gather by peer stores from inside the step kernel; "multicast" by one
    NVSwitch-multicast store per value (falls back to peer stores when the box has no multicast)."""
    shard.damping = float(damping)
    shard.setup_dangling(group)
    multi = dist.is_initialized() and dist.get_world_size(group) > 1
    pair = shard.enable_multicast_exchange(group) if (fused_exchange == "multicast" and multi) else None
    if pair is not None:
        r_a, r_b = pair
    elif fused_exchange and multi:
        r_a, r_b = shard.enable_peer_exchange(group)
    else:
        r_a = torch.empty(shard.n, dtype=torch.float32, device=shard.dev)
        r_b = torch.empty_like(r_a)
    partial = torch.zeros(3, dtype=torch.float64, device=shard.dev)
    shard.init_vector(r_a)
    fin, iters, residual, conv, l1 = pagerank_loop(shard, r_a, r_b, partial, bounds, damping, tolerance,
                                                    max_iterations, group, fixed_iterations)
    return PageRankOutcome(shard.normalize(fin), iters, residual, conv, l1)


# ------------------------------------------- native sharded PageRank (csrc/pagerank_dist.cu) ----
# The loop above (pagerank_loop / CudaShard) is the round-1 Python orchestration, kept for the
# backend-agnostic gloo tests.  The product path is the C++ one below: rendezvous, symmetric
# memory, multicast binding, in-kernel flag barrier and CUDA-graph replay all live in
# libspmv_b200.so; Python only passes pointers.

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
