// pagerank_dist.cu -- row-sharded PageRank over the GPUs of one NVSwitch box, host side in C++.
//
// The reference has no multi-GPU code (SURVEY 2, 8e); BASELINE.json config 5 / north_star ask for
// "PageRank on R-MAT 26 row-sharded across 8 B200, rank vector all-gathered, residual all-reduced".
// Signature family: pagerank() / PageRankConfig / PageRankResult, reference
// include/spmv/pagerank.h:9-32; recurrence and stop rule: reference src/pagerank.cu:93-150.
//
// Every rank owns a contiguous row shard (global column ids) and a FULL-length rank vector in a
// symmetric buffer (symm.hpp).  One iteration on a rank is a short chain of kernels on one stream,
// captured once in a CUDA graph and replayed:
//
//   gate     (1 warp)   waits until every rank has published iteration i-1 (flags in THIS rank's
//                       memory, written by the peers), adds the ranks' partial sums in rank order
//                       -> dangling mass for this iteration, and hands {sum d^2, sum |d|} of
//                       iteration i-1 to the host through mapped pinned memory
//   step     (pr_step)  the fused SpMV + damping/teleport/dangling/residual pass over the shard
//                       (csr_hot_kernels.cu / csr_merge_kernels.cu); finished rows are stored into
//                       EVERY rank's vector from inside the kernel: one multimem.st per value through
//                       the NVSwitch multicast mapping, or unicast peer stores
//   publish  (1 warp)   stores this rank's three partial sums into every rank's slot table, then --
//                       after a system-scope fence -- raises this rank's flag on every rank
//
// so the slice exchange ("all-gather") overlaps the product, the "all-reduce" of the three sums is
// N 24-byte peer stores + an ordered local sum, and no collective library call, host round trip or
// Python sits between two iterations.  The flag wait at the head of iteration i also covers the
// write-after-read hazard of the ping-pong vectors (nobody overwrites buffer (i+1)%2 of a rank that
// is still reading it in iteration i-1... it has published i-1 only after it finished reading).
//
// The literal north_star transport is kept as exchange mode NCCL: ncclBroadcast group (all-gather of
// uneven slices) + ncclAllGather of the 3-double partials, summed in rank order by the same gate
// kernel -- so all three modes produce bit-identical vectors (tests/test_gpu_multi.py, bench.py).
// NCCL is loaded with dlopen at first use: libspmv_b200.so has no link-time dependency on it.
//
// Stop rule: the reference's (L2 norm of the delta < tolerance, every iteration), read one iteration
// late exactly as in pagerank_device (pagerank.cu): the host polls the mapped history while the next
// iteration is already running.  Every rank sees the same sums, so every rank stops at the same
// iteration without talking to the others.
#include "pagerank_dist.hpp"

#include "internal.hpp"
#include "symm.hpp"

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

#include <dlfcn.h>

namespace spmv {
namespace b200 {
namespace {

// ---- layout of the symmetric control block ---------------------------------------------------
constexpr int kMaxRanks = kSymmMaxRanks;
struct ControlBlock {
    unsigned int flags[kMaxRanks];          // flags[p] = iterations rank p has published (written BY p)
    unsigned int pad0[8];
    double sums[2][kMaxRanks][3];           // [iteration parity][rank]{sum d^2, sum |d|, dangling mass}
};
struct LocalState {                         // plain device memory of one rank
    unsigned int epoch;                     // iterations this rank has published
    unsigned int pad[3];
    double total[3];                        // ordered sum over the ranks for the last gated iteration
};
struct HostHistoryEntry {
    double sums[3];
    volatile unsigned int ready;            // iteration number + 1 once the sums are valid
    unsigned int pad;
};

__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// One warp.  Waits for flags[p] >= epoch of every rank, then (epoch >= 1) folds the ranks' partial
// sums of iteration epoch-1 in rank order.  NCCL mode passes world_wait = 0 (stream order already
// guarantees the data) and reads the partials from `gathered` instead of the control block.
__global__ void pr_gate_kernel(const ControlBlock* __restrict__ ctl, LocalState* __restrict__ st, int world_wait,
                               int world, const double* __restrict__ gathered, float* __restrict__ d_dsum,
                               HostHistoryEntry* __restrict__ hist, int hist_cap, long long spin_limit) {
    const int lane = threadIdx.x;
    const unsigned int epoch = st->epoch;
    if (lane < world_wait) {
        long long spins = 0;
        while (ld_acquire_sys(ctl->flags + lane) < epoch) {
            if (++spins > spin_limit) break;  // a lost peer must not hang the GPU: the host sees stale history and fails
            __nanosleep(64);
        }
    }
    __syncwarp();
    if (lane == 0 && epoch >= 1) {
        const int parity = static_cast<int>((epoch - 1) & 1u);
        double t0 = 0.0, t1 = 0.0, t2 = 0.0;
        for (int p = 0; p < world; ++p) {
            const double* s = gathered ? gathered + 3 * p : ctl->sums[parity][p];
            t0 += *reinterpret_cast<const volatile double*>(s + 0);
            t1 += *reinterpret_cast<const volatile double*>(s + 1);
            t2 += *reinterpret_cast<const volatile double*>(s + 2);
        }
        st->total[0] = t0; st->total[1] = t1; st->total[2] = t2;
        *d_dsum = static_cast<float>(t2);  // dangling mass for the iteration about to start
        if (hist && static_cast<int>(epoch) <= hist_cap) {
            HostHistoryEntry* h = hist + (epoch - 1);
            h->sums[0] = t0; h->sums[1] = t1; h->sums[2] = t2;
            __threadfence_system();
            h->ready = epoch;
        }
    }
}

struct PeerControl {
    ControlBlock* peer[kMaxRanks];
};

// One warp, after the step: lane p stores this rank's partial sums into rank p's slot table, fences,
// and raises this rank's flag there.  All earlier kernels of the stream (whose peer / multicast
// stores carry the rank values) are complete before this kernel starts, and the release store
// orders them before the flag for any observer that acquires it.
__global__ void pr_publish_kernel(const double* __restrict__ partial, PeerControl peers, int world, int self,
                                  LocalState* __restrict__ st) {
    const int lane = threadIdx.x;
    const unsigned int epoch = st->epoch;
    const int parity = static_cast<int>(epoch & 1u);
    if (lane < world) {
        double* dst = peers.peer[lane]->sums[parity][self];
        dst[0] = partial[0]; dst[1] = partial[1]; dst[2] = partial[2];
        __threadfence_system();
        st_release_sys(peers.peer[lane]->flags + self, epoch + 1);
    }
    __syncwarp();
    if (lane == 0) st->epoch = epoch + 1;
}

// NCCL mode: no flags; just count the iteration
__global__ void pr_count_kernel(LocalState* __restrict__ st) {
    if (threadIdx.x == 0) st->epoch = st->epoch + 1;
}

// colsum_total[c] = sum over ranks (in rank order) of their local column sums, read through the
// peer mappings of a symmetric f64 scratch (set-up only)
struct PeerDoubles {
    const double* peer[kMaxRanks];
};
__global__ void pr_sum_peers_kernel(PeerDoubles src, int world, long long n, double* __restrict__ out) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        double t = 0.0;
        for (int p = 0; p < world; ++p) t += src.peer[p][i];
        out[i] = t;
    }
}

// ---- NCCL through dlopen ------------------------------------------------------------------------
struct NcclUniqueId { char internal[128]; };
typedef void* NcclComm;
struct NcclApi {
    bool ok = false;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(NcclComm*, int, NcclUniqueId, int) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*GetVersion)(int*) = nullptr;
};
constexpr int kNcclFloat32 = 7, kNcclFloat64 = 8;

const NcclApi& nccl() {
    static const NcclApi api = [] {
        NcclApi a;
        void* h = nullptr;
        const char* env = getenv("SPMV_B200_NCCL_LIB");
        const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) return a;
        auto sym = [&](const char* name) { return dlsym(h, name); };
        a.GetUniqueId = reinterpret_cast<int (*)(NcclUniqueId*)>(sym("ncclGetUniqueId"));
        a.CommInitRank = reinterpret_cast<int (*)(NcclComm*, int, NcclUniqueId, int)>(sym("ncclCommInitRank"));
        a.CommDestroy = reinterpret_cast<int (*)(NcclComm)>(sym("ncclCommDestroy"));
        a.Broadcast = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t)>(sym("ncclBroadcast"));
        a.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, NcclComm, cudaStream_t)>(sym("ncclAllGather"));
        a.GroupStart = reinterpret_cast<int (*)()>(sym("ncclGroupStart"));
        a.GroupEnd = reinterpret_cast<int (*)()>(sym("ncclGroupEnd"));
        a.GetVersion = reinterpret_cast<int (*)(int*)>(sym("ncclGetVersion"));
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.Broadcast && a.AllGather && a.GroupStart && a.GroupEnd;
        return a;
    }();
    return api;
}

}  // namespace

bool nccl_available() { return nccl().ok; }

// ---------------------------------------------------------------------------------- PrDist ----

struct PrDist {
    Comm* comm = nullptr;
    int rank = 0, world = 1;
    int exchange = kExchangeP2P;
    int n = 0, row_offset = 0, rows = 0;
    std::vector<int> bounds;  // world + 1 global row bounds
    PrPlan* plan = nullptr;
    cudaStream_t stream = nullptr;
    SymmBuffer r[2];          // the two full-length rank vectors
    SymmBuffer ctl;           // ControlBlock
    bool symmetric = false;   // r / ctl are symmetric buffers (else plain cudaMalloc: world == 1 or NCCL-only)
    float* plain_r[2] = {nullptr, nullptr};
    LocalState* d_state = nullptr;
    uint32_t* d_bits = nullptr;
    float* d_dsum = nullptr;
    double* d_partial = nullptr;   // this rank's {sum d^2, sum |d|, dangling}
    double* d_gathered = nullptr;  // NCCL mode: world x 3
    float* d_out = nullptr;        // normalised result (full length)
    float* d_pvec = nullptr;       // this shard's rows of the normalised personalization vector, or nullptr
    HostHistoryEntry* hist = nullptr;  // mapped pinned
    HostHistoryEntry* d_hist = nullptr;
    int hist_cap = 0;
    NcclComm nccl_comm = nullptr;
    PrIterationGraphs graphs;  // kept across runs
    bool dangling_ready = false;

    float* vec(int b) const { return symmetric ? static_cast<float*>(r[b].local) : plain_r[b]; }
};

namespace {

void free_all(PrDist* d) {
    if (!d) return;
    if (d->nccl_comm && nccl().ok) nccl().CommDestroy(d->nccl_comm);
    if (d->plan) pr_plan_destroy(d->plan);
    if (d->symmetric) {
        symm_free(&d->r[0]);
        symm_free(&d->r[1]);
        symm_free(&d->ctl);
    }
    cudaFree(d->plain_r[0]); cudaFree(d->plain_r[1]);
    cudaFree(d->d_state); cudaFree(d->d_bits); cudaFree(d->d_dsum); cudaFree(d->d_partial);
    cudaFree(d->d_gathered); cudaFree(d->d_out); cudaFree(d->d_pvec);
    if (d->hist) cudaFreeHost(d->hist);
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
}

bool agree(Comm* comm, bool mine) {
    std::vector<int> all(comm->world(), 0);
    const int v = mine ? 1 : 0;
    if (comm->allgather(&v, all.data(), sizeof(int)) != 0) return false;
    for (int x : all) if (!x) return false;
    return true;
}

// device-wide quiescence on every rank: nothing of an earlier run is still reading or writing
int global_quiesce(PrDist* d) {
    if (cudaStreamSynchronize(d->stream) != cudaSuccess) return -1;
    return d->comm->barrier();
}

}  // namespace

int pr_dist_create(Comm* comm, const CSRMatrix* shard, int row_offset, int n_global, int exchange, PrDist** out) {
    if (!comm || !shard || !out) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    const int world = comm->world(), rank = comm->rank();
    if (world > kMaxRanks || world > kMaxPeers) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    PrDist* d = new (std::nothrow) PrDist();
    if (!d) return static_cast<int>(SpMVError::OUT_OF_MEMORY);
    d->comm = comm; d->rank = rank; d->world = world;
    d->n = n_global; d->row_offset = row_offset; d->rows = shard->num_rows;

    // ---- shard bounds: contiguous, ordered, covering [0, n) ---------------------------------------
    int mine[2] = {row_offset, shard->num_rows};
    std::vector<int> all(2 * world);
    bool ok = comm->allgather(mine, all.data(), sizeof(mine)) == 0;
    d->bounds.assign(world + 1, 0);
    for (int p = 0; ok && p < world; ++p) {
        if (all[2 * p] != d->bounds[p]) ok = false;
        d->bounds[p + 1] = all[2 * p] + all[2 * p + 1];
    }
    if (ok && d->bounds[world] != n_global) ok = false;
    int rc = ok ? 0 : static_cast<int>(SpMVError::INVALID_DIMENSION);

    // ---- transport ----------------------------------------------------------------------------------
    if (exchange == kExchangeAuto) exchange = world > 1 ? kExchangeMulticast : kExchangeP2P;
    if (world == 1) exchange = kExchangeP2P;  // nothing to exchange
    const size_t vec_bytes = sizeof(float) * static_cast<size_t>(n_global > 0 ? n_global : 1);
    ok = rc == 0 && cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) == cudaSuccess;
    if (world > 1 && exchange != kExchangeNccl) {
        bool symm = ok && symm_supported();
        symm = agree(comm, symm);
        if (symm) {
            const bool want_mc = exchange == kExchangeMulticast && env_int("SPMV_B200_NO_MULTICAST", 0) == 0;
            bool a = symm_alloc(comm, vec_bytes, want_mc, &d->r[0]) == 0;
            bool b = a && symm_alloc(comm, vec_bytes, want_mc, &d->r[1]) == 0;
            bool c = b && symm_alloc(comm, sizeof(ControlBlock), false, &d->ctl) == 0;
            if (!(a && b && c)) {
                symm_free(&d->r[0]); symm_free(&d->r[1]); symm_free(&d->ctl);
                symm = false;
            }
        }
        if (symm) {
            d->symmetric = true;
            const bool mc = d->r[0].mc && d->r[1].mc;
            if (exchange == kExchangeMulticast && !mc) exchange = kExchangeP2P;  // box / driver without NVLS
        } else {
            exchange = kExchangeNccl;  // no peer mappings: fall back to the library collectives
        }
    }
    if (world > 1 && exchange == kExchangeNccl) {
        bool have = ok && nccl().ok;
        NcclUniqueId id;
        std::memset(&id, 0, sizeof(id));
        if (have && rank == 0) have = nccl().GetUniqueId(&id) == 0;
        std::vector<NcclUniqueId> ids(world);
        if (comm->allgather(&id, ids.data(), sizeof(id)) != 0) have = false;
        have = agree(comm, have);
        if (have) have = nccl().CommInitRank(&d->nccl_comm, world, ids[0], rank) == 0;
        have = agree(comm, have);
        if (!have) {
            ok = false;
            rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
        }
    }
    d->exchange = exchange;
    if (!d->symmetric) {
        ok = ok && cudaMalloc(&d->plain_r[0], vec_bytes) == cudaSuccess && cudaMalloc(&d->plain_r[1], vec_bytes) == cudaSuccess;
    }
    const size_t words = (static_cast<size_t>(n_global) + 31) / 32;
    d->hist_cap = 4096;
    ok = ok && cudaMalloc(&d->d_state, sizeof(LocalState)) == cudaSuccess &&
         cudaMalloc(&d->d_bits, sizeof(uint32_t) * (words ? words : 1)) == cudaSuccess &&
         cudaMalloc(&d->d_dsum, sizeof(float)) == cudaSuccess && cudaMalloc(&d->d_partial, 3 * sizeof(double)) == cudaSuccess &&
         cudaMalloc(&d->d_gathered, 3 * sizeof(double) * world) == cudaSuccess && cudaMalloc(&d->d_out, vec_bytes) == cudaSuccess &&
         cudaHostAlloc(&d->hist, sizeof(HostHistoryEntry) * d->hist_cap, cudaHostAllocMapped) == cudaSuccess &&
         cudaHostGetDevicePointer(&d->d_hist, d->hist, 0) == cudaSuccess;
    if (ok) {
        const int prc = pr_plan_create(shard, row_offset, n_global, d->stream, &d->plan);
        if (prc != 0) { ok = false; rc = prc; }
    }
    ok = ok && cudaStreamSynchronize(d->stream) == cudaSuccess;
    if (!agree(comm, ok)) {
        cudaGetLastError();
        free_all(d);
        return rc != 0 ? rc : static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    *out = d;
    return 0;
}

void pr_dist_destroy(PrDist* d) {
    if (!d) return;
    cudaStreamSynchronize(d->stream);
    d->comm->barrier();  // nobody unmaps a buffer a peer may still be storing into
    free_all(d);
}

int pr_dist_set_personalization(PrDist* d, const float* v_host) {
    if (!d) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (v_host) {  // the same host code on every rank: a vector one rank rejects, every rank rejects
        std::vector<float> vhat;
        const int rc = pr_personalization_normalise(v_host, d->n, &vhat);
        if (rc != 0) return rc;
    }
    // nothing of an earlier run still reads the old slice, and the cached iteration graphs, which hold its
    // address (or none), are dropped: the next run captures them again
    cudaStreamSynchronize(d->stream);
    d->graphs.reset();
    cudaFree(d->d_pvec);
    d->d_pvec = nullptr;
    int rc = pr_personalization_upload(v_host, d->n, d->row_offset, d->rows, &d->d_pvec, d->stream);
    if (!agree(d->comm, rc == 0)) {  // every rank runs the same form, or none keeps a vector
        cudaFree(d->d_pvec);
        d->d_pvec = nullptr;
        if (rc == 0) rc = static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    return rc;
}

int pr_dist_exchange(const PrDist* d) { return d ? d->exchange : -1; }
const float* pr_dist_ranks(const PrDist* d) { return d ? d->d_out : nullptr; }
cudaStream_t pr_dist_stream(const PrDist* d) { return d ? d->stream : nullptr; }
int pr_dist_hub_columns(const PrDist* d) { return d ? pr_plan_hub_columns(d->plan) : -1; }

namespace {

// dangling bitmask from the column sums of ALL shards (reference src/pagerank.cu:20-48): local f64
// sums into a symmetric scratch, ordered sum over the peers, bits.  Uses vector buffer 1 ... no:
// a dedicated symmetric f64 scratch, released afterwards (set-up only).
int setup_dangling(PrDist* d) {
    const size_t n = static_cast<size_t>(d->n);
    const CsrView& A = pr_plan_view(d->plan);
    bool ok = true;
    if (d->world == 1) {
        double* cs = nullptr;
        ok = cudaMalloc(&cs, sizeof(double) * (n ? n : 1)) == cudaSuccess &&
             pr_dangling_bits(A, cs, d->d_bits, d->stream) == cudaSuccess && cudaStreamSynchronize(d->stream) == cudaSuccess;
        cudaFree(cs);
        return ok ? 0 : -1;
    }
    if (d->symmetric) {
        SymmBuffer scratch;
        if (symm_alloc(d->comm, sizeof(double) * (n ? n : 1), false, &scratch) != 0) return -1;
        double* total = nullptr;
        ok = cudaMalloc(&total, sizeof(double) * (n ? n : 1)) == cudaSuccess;
        if (ok) {
            cudaMemsetAsync(scratch.local, 0, sizeof(double) * n, d->stream);
            ok = launch_colsum(A, static_cast<double*>(scratch.local), d->stream) == cudaSuccess &&
                 cudaStreamSynchronize(d->stream) == cudaSuccess;
        }
        ok = agree(d->comm, ok);  // also the barrier: every rank's local sums are complete
        if (ok) {
            PeerDoubles src;
            for (int p = 0; p < kMaxRanks; ++p) src.peer[p] = p < d->world ? static_cast<const double*>(scratch.peer[p]) : nullptr;
            pr_sum_peers_kernel<<<148 * 8, 256, 0, d->stream>>>(src, d->world, static_cast<long long>(n), total);
            count_launches(1);
            ok = launch_dangling_bits(total, d->n, d->n, d->d_bits, d->stream) == cudaSuccess &&
                 cudaStreamSynchronize(d->stream) == cudaSuccess;
        }
        ok = agree(d->comm, ok);  // nobody frees its scratch while a peer still reads it
        cudaFree(total);
        symm_free(&scratch);
        return ok ? 0 : -1;
    }
    // NCCL only: all-gather the local sums chunk-wise and add them in rank order
    const size_t chunk = 1u << 22;
    double *local = nullptr, *gath = nullptr, *total = nullptr;
    ok = cudaMalloc(&local, sizeof(double) * (n ? n : 1)) == cudaSuccess &&
         cudaMalloc(&gath, sizeof(double) * chunk * d->world) == cudaSuccess &&
         cudaMalloc(&total, sizeof(double) * (n ? n : 1)) == cudaSuccess;
    if (ok) {
        cudaMemsetAsync(local, 0, sizeof(double) * n, d->stream);
        ok = launch_colsum(A, local, d->stream) == cudaSuccess;
    }
    ok = agree(d->comm, ok);
    for (size_t lo = 0; ok && lo < n; lo += chunk) {
        // every rank contributes `chunk` doubles (the last chunk reads past n inside the padded scratch: sized n, so clamp)
        const size_t len = n - lo < chunk ? n - lo : chunk;
        ok = nccl().AllGather(local + lo, gath, len, kNcclFloat64, d->nccl_comm, d->stream) == 0;
        if (!ok) break;
        PeerDoubles src;
        for (int p = 0; p < kMaxRanks; ++p) src.peer[p] = p < d->world ? gath + static_cast<size_t>(p) * len : nullptr;
        pr_sum_peers_kernel<<<148 * 4, 256, 0, d->stream>>>(src, d->world, static_cast<long long>(len), total + lo);
        count_launches(1);
    }
    if (ok) ok = launch_dangling_bits(total, d->n, d->n, d->d_bits, d->stream) == cudaSuccess;
    ok = cudaStreamSynchronize(d->stream) == cudaSuccess && ok;
    cudaFree(local); cudaFree(gath); cudaFree(total);
    return agree(d->comm, ok) ? 0 : -1;
}

// one iteration from vector buffer `from` into the other one, enqueued on d->stream
int enqueue_iteration(PrDist* d, int from, float damping) {
    const int to = from ^ 1;
    const bool fused = d->world > 1 && d->exchange != kExchangeNccl;
    const ControlBlock* ctl = d->symmetric ? static_cast<const ControlBlock*>(d->ctl.local) : nullptr;
    static const long long spin_limit = static_cast<long long>(env_int("SPMV_B200_GATE_SPIN_LIMIT", 200000000));
    pr_gate_kernel<<<1, 32, 0, d->stream>>>(ctl, d->d_state, fused ? d->world : 0, d->world,
                                            fused ? nullptr : d->d_gathered, d->d_dsum, d->d_hist, d->hist_cap, spin_limit);
    count_launches(1);
    float* peers[kMaxPeers] = {};
    float* mc = nullptr;
    if (fused) {
        for (int p = 0; p < d->world; ++p) peers[p] = static_cast<float*>(d->r[to].peer[p]);
        if (d->exchange == kExchangeMulticast) mc = static_cast<float*>(d->r[to].mc);
    }
    int rc = pr_step(d->plan, d->vec(from), d->vec(to), damping, d->d_dsum, d->d_bits, d->d_partial, d->stream,
                     fused ? peers : nullptr, fused ? d->world : 0, d->rank, mc, d->d_pvec);
    if (rc != 0) return rc;
    if (fused) {
        PeerControl pc;
        for (int p = 0; p < kMaxRanks; ++p) pc.peer[p] = p < d->world ? static_cast<ControlBlock*>(d->ctl.peer[p]) : nullptr;
        pr_publish_kernel<<<1, 32, 0, d->stream>>>(d->d_partial, pc, d->world, d->rank, d->d_state);
        count_launches(1);
    } else {
        if (d->world > 1) {
            const NcclApi& N = nccl();
            float* v = d->vec(to);
            bool ok = N.GroupStart() == 0;
            for (int p = 0; ok && p < d->world; ++p) {
                const size_t cnt = static_cast<size_t>(d->bounds[p + 1] - d->bounds[p]);
                if (cnt) ok = N.Broadcast(v + d->bounds[p], v + d->bounds[p], cnt, kNcclFloat32, p, d->nccl_comm, d->stream) == 0;
            }
            ok = N.GroupEnd() == 0 && ok;
            ok = ok && N.AllGather(d->d_partial, d->d_gathered, 3, kNcclFloat64, d->nccl_comm, d->stream) == 0;
            if (!ok) return static_cast<int>(SpMVError::KERNEL_LAUNCH);
        } else {
            cudaMemcpyAsync(d->d_gathered, d->d_partial, 3 * sizeof(double), cudaMemcpyDeviceToDevice, d->stream);
        }
        pr_count_kernel<<<1, 32, 0, d->stream>>>(d->d_state);
        count_launches(1);
    }
    return cudaGetLastError() == cudaSuccess ? 0 : static_cast<int>(SpMVError::KERNEL_LAUNCH);
}

// the gate alone: publishes the sums of the last iteration to the host history
void enqueue_final_gate(PrDist* d) {
    const bool fused = d->world > 1 && d->exchange != kExchangeNccl;
    const ControlBlock* ctl = d->symmetric ? static_cast<const ControlBlock*>(d->ctl.local) : nullptr;
    pr_gate_kernel<<<1, 32, 0, d->stream>>>(ctl, d->d_state, fused ? d->world : 0, d->world,
                                            fused ? nullptr : d->d_gathered, d->d_dsum, d->d_hist, d->hist_cap, 200000000LL);
    count_launches(1);
}

bool wait_history(PrDist* d, int iteration /* 1-based */, double timeout_s) {
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::duration<double>(timeout_s);
    volatile unsigned int* ready = &d->hist[iteration - 1].ready;
    int spins = 0;
    while (*ready != static_cast<unsigned int>(iteration)) {
        if (++spins > 2000) {
            if (cudaStreamQuery(d->stream) != cudaErrorNotReady && *ready != static_cast<unsigned int>(iteration)) {
                // the stream drained (or failed) without publishing: give the write a moment, then give up
                std::this_thread::sleep_for(std::chrono::milliseconds(1));
                if (*ready != static_cast<unsigned int>(iteration)) return false;
            }
            if (std::chrono::steady_clock::now() > deadline) return false;
            spins = 0;
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    return true;
}

}  // namespace

int pr_dist_run(PrDist* d, const PageRankConfig* config, int fixed_iterations, PrDistResult* out) {
    NvtxRange nvtx_range("spmv_b200:pagerank_multi.run");
    if (!d || !out) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    PageRankConfig defaults;
    if (!config) config = &defaults;
    *out = PrDistResult();
    out->exchange = d->exchange;
    const int limit = fixed_iterations > 0 ? fixed_iterations : config->max_iterations;
    if (d->n <= 0 || limit <= 0) return 0;
    if (limit > d->hist_cap) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    int rc = 0;

    if (!d->dangling_ready) {
        if (setup_dangling(d) != 0) return static_cast<int>(SpMVError::KERNEL_LAUNCH);
        d->dangling_ready = true;
    }
    // ---- reset: nothing of an earlier run may still be in flight anywhere ------------------------
    if (global_quiesce(d) != 0) return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    std::memset(d->hist, 0, sizeof(HostHistoryEntry) * d->hist_cap);
    cudaMemsetAsync(d->d_state, 0, sizeof(LocalState), d->stream);
    if (d->symmetric) cudaMemsetAsync(d->ctl.local, 0, sizeof(ControlBlock), d->stream);
    cudaMemsetAsync(d->d_gathered, 0, 3 * sizeof(double) * d->world, d->stream);
    launch_pr_init(d->n, d->d_bits, d->vec(0), d->d_dsum, pr_plan_tmp(d->plan), d->stream);
    if (global_quiesce(d) != 0) return static_cast<int>(SpMVError::KERNEL_LAUNCH);

    // ---- CUDA graphs of the two ping-pong iterations (fused modes; NCCL calls stay eager) ----------
    const bool fused = d->world == 1 || d->exchange != kExchangeNccl;
    if (fused && !d->graphs.ready() && PrIterationGraphs::wanted(limit))
        d->graphs.capture(d->stream, [&](int p) { return enqueue_iteration(d, p, config->damping_factor); });
    // every rank replays or none does (a rank that failed to capture would still work, but keep the
    // launch pattern identical everywhere)
    const bool replay = agree(d->comm, d->graphs.ready());

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEventCreate(&ev0);
    cudaEventCreate(&ev1);
    d->comm->barrier();
    const auto wall0 = std::chrono::steady_clock::now();
    cudaEventRecord(ev0, d->stream);

    int iters = 0, launched = 0;
    float residual = 0.0f;
    double l1 = 0.0;
    bool conv = false;
    int final_buf = 0;  // buffer holding the final iterate
    const double timeout_s = static_cast<double>(env_int("SPMV_B200_PR_TIMEOUT_S", 120));
    auto settle = [&](int iteration) -> bool {  // true when that iteration met the tolerance
        if (!wait_history(d, iteration, timeout_s)) {
            rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
            return true;
        }
        residual = std::sqrt(static_cast<float>(d->hist[iteration - 1].sums[0]));  // reference :118
        l1 = d->hist[iteration - 1].sums[1];
        iters = iteration;
        final_buf = iteration & 1;  // iteration k reads buffer (k-1)&1 and writes k&1
        return fixed_iterations <= 0 && residual < config->tolerance;
    };
    for (int it = 0; it < limit; ++it) {
        const int from = it & 1;
        if (replay) {
            if (!d->graphs.launch(from, d->stream)) {
                rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
                break;
            }
        } else {
            rc = enqueue_iteration(d, from, config->damping_factor);
            if (rc != 0) break;
        }
        ++launched;
        // the sums of iteration `it` (1-based) are published by the gate of iteration it + 1, which is
        // queued right above: the host inspects them while that iteration runs
        if (it >= 1 && settle(it)) {
            conv = rc == 0;
            break;
        }
    }
    if (!conv && rc == 0) {
        enqueue_final_gate(d);
        conv = settle(launched) && fixed_iterations <= 0 && rc == 0;
    }
    cudaEventRecord(ev1, d->stream);
    cudaError_t e = cudaStreamSynchronize(d->stream);  // a speculative iteration may still be running
    const auto wall1 = std::chrono::steady_clock::now();
    float ms = 0.0f;
    if (e == cudaSuccess) cudaEventElapsedTime(&ms, ev0, ev1);
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (rc == 0) rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    // everybody has left the loop before anyone touches the vectors again
    if (!agree(d->comm, rc == 0) && rc == 0) rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
    if (rc == 0) {
        launch_normalize(d->vec(final_buf), d->n, d->d_out, pr_plan_tmp(d->plan), d->stream);
        if (cudaStreamSynchronize(d->stream) != cudaSuccess) {
            cudaGetLastError();
            rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
        }
    }
    out->iterations = iters;
    out->final_residual = residual;
    out->converged = conv ? 1 : 0;
    out->l1_residual = l1;
    out->iterations_launched = launched;
    out->device_seconds = ms * 1e-3;
    out->wall_seconds = std::chrono::duration<double>(wall1 - wall0).count();
    out->graph_replay = replay ? 1 : 0;
    out->kernels_per_iteration = static_cast<int>(d->graphs.launches_per_iteration);
    return rc;
}

}  // namespace b200
}  // namespace spmv
