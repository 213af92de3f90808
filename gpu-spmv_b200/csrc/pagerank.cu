// pagerank.cu -- PageRank on the fused merge-path iteration.
//
// Replaces pagerank() (reference src/pagerank.cu:50-153).  The reference runs
// only the SpMV on the GPU and, EVERY iteration, copies the rank vector to the
// host, applies damping/teleport/dangling mass there with single-threaded fp32
// loops, copies it back and computes the L2 residual on the host.  Here the
// whole iteration is one pass of merge_tile_kernel<PageRankRow> (+ its fix-up
// and a 1-CTA reduction): the rank vectors never leave HBM and the only
// per-iteration host traffic is the 24-byte {sum d^2, sum |d|, dangling mass}.
//
// Recurrence, initial vector, update expression order, stop rule (L2 norm of
// the delta < tolerance, checked after every iteration), result fields and the
// final normalisation follow the reference line by line; the three global
// sums use f64 accumulators because the reference's sequential fp32 host sums
// lose all accuracy at n = 2^26 (SURVEY F7).
//
// The same building blocks work on a row shard of the matrix (row_offset,
// n_global) so that one process per GPU can run a sharded PageRank with an
// all-gather of the rank slices and an all-reduce of the three sums in between
// (gpu-spmv_b200/dist.py).
#include "internal.hpp"

#include <cmath>
#include <new>

namespace spmv {
namespace b200 {

// A plan over one row shard: merge-path coordinates are computed once (the
// matrix is constant across iterations) and the work arrays are owned here.
struct PrPlan {
    CsrView A{};
    int row_offset = 0;
    int n_global = 0;
    Scratch merge_block;
    MergePlan merge;
    Scratch tmp_block;   // kPrScratchDoubles doubles
    double* tmp = nullptr;
    // A ROW SHARD of a scale-free graph takes the hub-column plan: the tile epilogue of that kernel
    // overlaps the slice exchange with the product (8 GPUs, R-MAT 26: 1.17 vs 1.46 ms per iteration
    // against the segmented-stream kernel, whose exchange is a separate pass).  The WHOLE graph on
    // one GPU has nothing to exchange and takes the segmented stream with its streaming epilogue
    // (R-MAT 26: 5.45 vs 5.89 ms per iteration; R-MAT 24: 1.21 vs 1.29).  Neither: plain tile kernel.
    PlannedCsr planned;
    bool whole_graph = false;
    ~PrPlan() { planned.release(); }
};

int pr_plan_create(const CSRMatrix* shard, int row_offset, int n_global, cudaStream_t stream, PrPlan** out) {
    if (!shard || !out || row_offset < 0 || n_global < 0) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (static_cast<long long>(row_offset) + shard->num_rows > n_global)
        return static_cast<int>(SpMVError::INVALID_DIMENSION);
    // every kernel gathers r[col] for col < num_cols from a rank vector of n_global entries: a shard (or a whole
    // adjacency matrix) with another column count would read past it.  The reference rejects the same input in
    // spmv_csr(..., vec_size = n) -> INVALID_DIMENSION (src/spmv_kernels.cu:224-226, src/pagerank.cu:102-107).
    if (shard->num_cols != n_global) return static_cast<int>(SpMVError::INVALID_DIMENSION);
    if (!shard->d_row_ptrs || (shard->nnz > 0 && (!shard->d_col_indices || !shard->d_values)))
        return static_cast<int>(SpMVError::INVALID_FORMAT);
    PrPlan* p = new (std::nothrow) PrPlan();
    if (!p) return static_cast<int>(SpMVError::OUT_OF_MEMORY);
    p->A = view_of(shard);
    p->row_offset = row_offset;
    p->n_global = n_global;
    void* block = p->merge_block.reserve(merge_plan_bytes(p->A.rows, p->A.nnz, true));
    p->tmp = static_cast<double*>(p->tmp_block.reserve(kPrScratchDoubles * sizeof(double)));
    if (!block || !p->tmp) {
        delete p;
        return static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    p->merge = merge_plan_carve(block, p->A.rows, p->A.nnz, true);
    if (p->A.rows > 0 && launch_merge_partition(p->A, p->merge, stream) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    // the matrix is constant over the iterations: the hub-column plan pays for itself after a few
    p->whole_graph = row_offset == 0 && shard->num_rows == n_global;
    if (hot_env_mode() != 0 &&
        planned_build(p->A, &p->planned, 0, hot_env_mode() > 0, p->whole_graph, stream, p->whole_graph) != cudaSuccess) {
        cudaGetLastError();
        p->planned.release();  // not fatal: the plain tile kernel is used
    }
    *out = p;
    return 0;
}

void pr_plan_destroy(PrPlan* p) { delete p; }

// max_hot_columns: 0 drops the plan (plain tile kernel), < 0 device maximum; force skips the
// size / benefit thresholds.  Returns the number of hub columns now in use, or a negative error.
int pr_plan_set_hot(PrPlan* p, int max_hot_columns, bool force, cudaStream_t stream) {
    if (!p) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    cudaStreamSynchronize(stream);
    p->planned.release();
    if (max_hot_columns == 0) return 0;
    if (planned_build(p->A, &p->planned, max_hot_columns < 0 ? 0 : max_hot_columns, force, p->whole_graph, stream,
                      p->whole_graph) != cudaSuccess) {
        cudaGetLastError();
        p->planned.release();
        return static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    return p->planned.seg.valid() ? (p->planned.seg.n_hot > 0 ? p->planned.seg.n_hot : 1) : p->planned.hot.n_hot;
}

int pr_step(PrPlan* p, const float* d_r_old, float* d_r_new, float damping, const float* d_dsum,
            const uint32_t* d_bits, double* d_partial, cudaStream_t stream, float* const* peer_r_new, int n_peers,
            int self_rank, float* mc_r_new, const float* d_pvec) {
    if (!p || !d_r_old || !d_r_new || !d_dsum || !d_bits || !d_partial)
        return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (n_peers > kMaxPeers || (n_peers > 1 && ((!peer_r_new && !mc_r_new) || self_rank < 0 || self_rank >= n_peers)))
        return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    PageRankStepArgs a;
    a.n_peers = n_peers > 1 ? n_peers : 0;
    a.self_rank = self_rank;
    for (int i = 0; i < kMaxPeers; ++i) a.peers[i] = (n_peers > 1 && i < n_peers && peer_r_new) ? peer_r_new[i] : nullptr;
    a.mc_r_new = n_peers > 1 ? mc_r_new : nullptr;
    a.r_old = d_r_old;
    a.r_new = d_r_new;
    a.row_offset = p->row_offset;
    a.n_global = p->n_global;
    a.damping = damping;
    a.teleport = d_pvec ? 1.0f - damping : (1.0f - damping) / p->n_global;  // reference src/pagerank.cu:86
    a.pvec = d_pvec;
    a.d_dsum = d_dsum;
    a.bits = d_bits;
    a.out = d_partial;
    const cudaError_t e = p->planned.seg.valid()     ? launch_seg_pagerank(p->A, p->planned.seg, a, stream)
                          : p->planned.hot.n_hot > 0 ? launch_hot_pagerank(p->A, p->planned.hot, p->merge, a, stream)
                                                     : launch_merge_pagerank(p->A, p->merge, a, stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

const CsrView& pr_plan_view(const PrPlan* p) { return p->A; }
int pr_plan_hub_columns(const PrPlan* p) {
    if (!p) return 0;
    return p->planned.seg.valid() ? p->planned.seg.n_hot : p->planned.hot.n_hot;
}
double* pr_plan_tmp(PrPlan* p) { return p->tmp; }

cudaError_t pr_dangling_bits(const CsrView& A, double* d_colsum, uint32_t* d_bits, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(d_colsum, 0, sizeof(double) * A.cols, stream);
    if (e == cudaSuccess) e = launch_colsum(A, d_colsum, stream);
    if (e == cudaSuccess) e = launch_dangling_bits(d_colsum, A.cols, A.cols, d_bits, stream);
    return e;
}

bool PrIterationGraphs::wanted(int iterations) {
    static const int enabled = env_int("SPMV_B200_PR_GRAPH", 1);
    return enabled && iterations >= 4;
}

bool PrIterationGraphs::capture(cudaStream_t stream, const std::function<int(int)>& enqueue) {
    for (int p = 0; p < 2; ++p) {
        cudaGraph_t g = nullptr;
        const unsigned long long before = launch_count();
        bool good = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (good) {
            const int r = enqueue(p);
            good = cudaStreamEndCapture(stream, &g) == cudaSuccess && r == 0 && g != nullptr;
        }
        launches_per_iteration = launch_count() - before;
        count_launches(-static_cast<int>(launches_per_iteration));  // captured, not launched
        if (good) good = cudaGraphInstantiate(&exec[p], g, 0) == cudaSuccess;
        if (g) cudaGraphDestroy(g);
        if (!good) {
            cudaGetLastError();
            reset();
            return false;
        }
    }
    return true;
}

bool PrIterationGraphs::launch(int p, cudaStream_t stream) {
    if (cudaGraphLaunch(exec[p], stream) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    count_launches(static_cast<int>(launches_per_iteration));
    return true;
}

void PrIterationGraphs::reset() {
    for (int p = 0; p < 2; ++p) {
        if (exec[p]) cudaGraphExecDestroy(exec[p]);
        exec[p] = nullptr;
    }
}

// pagerank_small.cu
bool pagerank_small_applies(int n, int nnz);
cudaError_t pagerank_small_run(const CsrView& A, float damping, float tolerance, int max_iterations, const uint32_t* d_bits,
                               float* buf_a, float* buf_b, const float* d_dsum, float* l2_history, int history_capacity,
                               int* iterations, float* residual, double* l1, bool* converged, int* final_buffer,
                               cudaStream_t stream, const float* d_pvec);

// What one single-GPU run allocates, freed on every return.  init() sets up what both loops start from; the
// multi-kernel loop adds its plan and the two copies of the per-iteration sums.
struct PrRun {
    float *a = nullptr, *b = nullptr;  // the rank vectors; a holds r_0
    double* colsum = nullptr;
    uint32_t* bits = nullptr;          // dangling bitmask
    float* dsum = nullptr;             // dangling mass of r_0
    double* tmp = nullptr;             // kPrScratchDoubles, for pr_init and normalize
    PrPlan* plan = nullptr;
    double* partial = nullptr;         // device {sum d^2, sum |d|, dangling mass} of one iteration
    double* h_partial = nullptr;       // pinned, one triple per ping-pong slot
    PrRun() = default;
    PrRun(const PrRun&) = delete;
    PrRun& operator=(const PrRun&) = delete;
    ~PrRun() {
        cudaFree(a); cudaFree(b); cudaFree(colsum); cudaFree(bits); cudaFree(dsum); cudaFree(tmp); cudaFree(partial);
        if (h_partial) cudaFreeHost(h_partial);
        pr_plan_destroy(plan);
    }
    // dangling nodes, r_0 = 1/n and its dangling mass (reference :20-48, :69-72, :87, :94-99 for iteration 0)
    int init(const CsrView& A, cudaStream_t stream) {
        const int n = A.rows;
        const size_t words = (static_cast<size_t>(n) + 31) / 32;
        if (cudaMalloc(&a, sizeof(float) * n) != cudaSuccess || cudaMalloc(&b, sizeof(float) * n) != cudaSuccess ||
            cudaMalloc(&colsum, sizeof(double) * n) != cudaSuccess || cudaMalloc(&bits, sizeof(uint32_t) * words) != cudaSuccess ||
            cudaMalloc(&dsum, sizeof(float)) != cudaSuccess || cudaMalloc(&tmp, sizeof(double) * kPrScratchDoubles) != cudaSuccess) {
            cudaGetLastError();
            return static_cast<int>(SpMVError::CUDA_MALLOC);
        }
        if (pr_dangling_bits(A, colsum, bits, stream) != cudaSuccess || launch_pr_init(n, bits, a, dsum, tmp, stream) != cudaSuccess) {
            cudaGetLastError();
            return static_cast<int>(SpMVError::KERNEL_LAUNCH);
        }
        return 0;
    }
    // final vector (:135-139) into d_ranks, normalised (:142-150) or raw; the stream is synchronised
    int write_ranks(const float* fin, int n, bool normalize, float* d_ranks, cudaStream_t stream) {
        if (normalize) launch_normalize(fin, n, d_ranks, tmp, stream);
        else cudaMemcpyAsync(d_ranks, fin, sizeof(float) * n, cudaMemcpyDeviceToDevice, stream);
        if (cudaStreamSynchronize(stream) == cudaSuccess) return 0;
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
};

// The whole loop on one device; d_ranks receives the ranks, normalised on the device with an
// f64 sum when `normalize` is set, else the raw final iterate.
int pagerank_device(const CSRMatrix* adj, const PageRankConfig* config, float* d_ranks, int* iterations,
                    float* final_residual, bool* converged, double* l1_residual, bool normalize, float* l2_history,
                    int history_capacity, const float* d_pvec) {
    NvtxRange nvtx_range("spmv_b200:pagerank_device");
    if (!adj || !d_ranks) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    PageRankConfig defaults;
    if (!config) config = &defaults;
    const int n = adj->num_rows;
    if (iterations) *iterations = 0;
    if (final_residual) *final_residual = 0.0f;
    if (converged) *converged = false;
    if (l1_residual) *l1_residual = 0.0;
    if (n <= 0) return 0;
    // non-square adjacency: the reference's first spmv_csr(adj, ..., vec_size = n) fails with INVALID_DIMENSION and
    // pagerank() returns the uniform vector with iterations = 0 (src/pagerank.cu:102-107); pagerank() below does the same
    if (adj->num_cols != n) return static_cast<int>(SpMVError::INVALID_DIMENSION);
    if (!adj->d_row_ptrs || (adj->nnz > 0 && (!adj->d_col_indices || !adj->d_values)))
        return static_cast<int>(SpMVError::INVALID_FORMAT);

    cudaStream_t stream = nullptr;
    PrRun run;
    int rc = run.init(view_of(adj), stream);
    if (rc != 0) return rc;

    if (pagerank_small_applies(n, adj->nnz)) {  // launch-bound sizes: the whole loop in one persistent kernel
        int fin = 0;
        const cudaError_t e = pagerank_small_run(view_of(adj), config->damping_factor, config->tolerance, config->max_iterations,
                                                 run.bits, run.a, run.b, run.dsum, l2_history, history_capacity, iterations,
                                                 final_residual, l1_residual, converged, &fin, stream, d_pvec);
        if (e == cudaSuccess) return run.write_ranks(fin ? run.b : run.a, n, normalize, d_ranks, stream);
        if (e != cudaErrorNotSupported) {
            cudaGetLastError();
            return static_cast<int>(SpMVError::KERNEL_LAUNCH);
        }
        // no cooperative launch on this device: the multi-kernel loop below, on the same (untouched) buffers
    }

    rc = pr_plan_create(adj, 0, n, stream, &run.plan);
    if (rc != 0) return rc;
    if (cudaMalloc(&run.partial, 3 * sizeof(double)) != cudaSuccess ||
        cudaMallocHost(&run.h_partial, 6 * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::CUDA_MALLOC);
    }

    // The stop rule is the reference's (L2 norm of the delta < tolerance, every iteration,
    // :118-127) but it is read one iteration late: the 24-byte sums of iteration i go to pinned
    // host memory asynchronously and are inspected while iteration i+1 is already queued, so the
    // device never idles on the host.  If iteration i had converged, its output is the INPUT of
    // the speculative iteration i+1 (which writes the other buffer), so vector, iteration count
    // and residual are exactly those of the eager rule.
    float* r_old = run.a;
    float* r_new = run.b;
    const float* fin = r_old;  // what the reference returns when the loop never runs (:135-139)
    int iters = 0;
    float residual = 0.0f;
    double l1 = 0.0;
    bool conv = false;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
    struct Pending { int iter; int slot; const float* vec; bool valid; } pending = {0, 0, nullptr, false};
    auto settle = [&](const Pending& p) -> bool {  // true when that iteration met the tolerance
        if (cudaEventSynchronize(ev[p.slot]) != cudaSuccess) {
            cudaGetLastError();
            rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
            return true;
        }
        residual = std::sqrt(static_cast<float>(run.h_partial[3 * p.slot + 0]));  // L2 norm of the delta (:118)
        l1 = run.h_partial[3 * p.slot + 1];
        iters = p.iter;
        if (l2_history && p.iter >= 1 && p.iter <= history_capacity) l2_history[p.iter - 1] = residual;
        fin = p.vec;
        return residual < config->tolerance;  // :123-127
    };
    // One iteration = the fused step (3-4 kernels), the dangling-mass hand-over and the 24-byte download.
    auto enqueue_iteration = [&](float* from, float* to, int slot, cudaStream_t s) -> int {
        const int r = pr_step(run.plan, from, to, config->damping_factor, run.dsum, run.bits, run.partial, s, nullptr, 0, 0,
                              nullptr, d_pvec);
        if (r != 0) return r;
        launch_next_dsum(run.partial, run.dsum, s);
        cudaMemcpyAsync(run.h_partial + 3 * slot, run.partial, 3 * sizeof(double), cudaMemcpyDeviceToHost, s);
        return 0;
    };
    // Graph replay (SURVEY 8f rank 3); the stop rule stays per iteration (above).  Capture needs a real
    // stream; a blocking one keeps the legacy default stream's ordering.  Any failure falls back to the
    // eager loop.
    cudaStream_t gs = nullptr;
    PrIterationGraphs graphs;
    if (PrIterationGraphs::wanted(config->max_iterations) && cudaStreamCreate(&gs) == cudaSuccess)
        graphs.capture(gs, [&](int p) { return enqueue_iteration(p ? run.b : run.a, p ? run.a : run.b, p, gs); });
    const bool replay = graphs.ready();
    cudaStream_t loop_stream = replay ? gs : stream;
    for (int it = 0; it < config->max_iterations; ++it) {
        const int slot = it & 1;
        if (replay) {
            if (!graphs.launch(slot, gs)) {
                rc = static_cast<int>(SpMVError::KERNEL_LAUNCH);
                break;
            }
        } else {
            rc = enqueue_iteration(r_old, r_new, slot, stream);
            if (rc != 0) break;  // the reference also leaves the loop on a failed SpMV (:105-107)
        }
        cudaEventRecord(ev[slot], loop_stream);
        if (pending.valid) {
            const bool done = settle(pending);
            pending.valid = false;
            if (done) {
                conv = rc == 0;
                break;
            }
        }
        pending = {it + 1, slot, r_new, true};
        float* t = r_old; r_old = r_new; r_new = t;  // :130-131
    }
    if (pending.valid && rc == 0) conv = settle(pending) && rc == 0;
    cudaEventDestroy(ev[0]);
    cudaEventDestroy(ev[1]);
    if (gs) {
        cudaStreamSynchronize(gs);  // a speculative iteration may still be running
        cudaStreamDestroy(gs);
    }
    const int wr = run.write_ranks(fin, n, normalize, d_ranks, stream);
    if (rc == 0) rc = wr;
    if (iterations) *iterations = iters;
    if (final_residual) *final_residual = residual;
    if (converged) *converged = conv;
    if (l1_residual) *l1_residual = l1;
    return rc;
}

int pr_personalization_normalise(const float* v, int n, std::vector<float>* vhat) {
    if (!v || n <= 0 || !vhat) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    double sum = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!std::isfinite(v[i]) || v[i] < 0.0f) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
        sum += static_cast<double>(v[i]);
    }
    if (sum == 0.0) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    vhat->resize(static_cast<size_t>(n));
    for (int i = 0; i < n; ++i) (*vhat)[i] = static_cast<float>(static_cast<double>(v[i]) / sum);
    return 0;
}

int pr_personalization_upload(const float* v, int n, int row_lo, int rows, float** d_out, cudaStream_t stream) {
    if (!d_out || row_lo < 0 || rows < 0 || static_cast<long long>(row_lo) + rows > n)
        return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    *d_out = nullptr;
    if (!v) return 0;
    std::vector<float> vhat;
    const int rc = pr_personalization_normalise(v, n, &vhat);
    if (rc != 0) return rc;
    float* d = nullptr;
    if (cudaMalloc(&d, sizeof(float) * static_cast<size_t>(rows > 0 ? rows : 1)) != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    // synchronised: vhat is freed on return, and the kernels that read d may run on another stream
    if (rows > 0 && (cudaMemcpyAsync(d, vhat.data() + row_lo, sizeof(float) * static_cast<size_t>(rows), cudaMemcpyHostToDevice,
                                     stream) != cudaSuccess ||
                     cudaStreamSynchronize(stream) != cudaSuccess)) {
        cudaGetLastError();
        cudaFree(d);
        return static_cast<int>(SpMVError::CUDA_MEMCPY);
    }
    *d_out = d;
    return 0;
}

// API-compatible body of pagerank(): result->ranks is a host new[] array (pagerank_free
// deletes it).  adj must already be on the device; unlike the reference the
// host arrays are not needed (the dangling scan runs on the device).
int pagerank_to_host(const CSRMatrix* adj_matrix, const PageRankConfig* config, const float* personalization,
                     PageRankResult* out) {
    PageRankResult& result = *out;
    if (!adj_matrix) return personalization ? static_cast<int>(SpMVError::INVALID_ARGUMENT) : 0;
    const int n = adj_matrix->num_rows;
    float* d_pvec = nullptr;
    if (personalization) {  // validated before anything touches the device
        const int rc = pr_personalization_upload(personalization, n, 0, n, &d_pvec, nullptr);
        if (rc != 0) return rc;
    }
    try {
        result.ranks = new float[n > 0 ? n : 0];
    } catch (...) {
        cudaFree(d_pvec);
        throw;
    }
    if (n <= 0) return 0;

    // the reference's final normalisation (:142-150): sequential fp32 sum, then every entry divided by it
    auto normalise_literally = [&]() {
        float sum = 0.0f;
        for (int i = 0; i < n; ++i) sum += result.ranks[i];
        if (sum > 0.0f)
            for (int i = 0; i < n; ++i) result.ranks[i] /= sum;
    };

    float* d_ranks = nullptr;
    if (cudaMalloc(&d_ranks, sizeof(float) * n) != cudaSuccess) {
        cudaFree(d_pvec);
        throw CudaException(cudaGetLastError());
    }
    int iters = 0;
    float residual = 0.0f;
    bool conv = false;
    // Up to 2^24 nodes the final normalisation is the reference's own host code (sequential fp32
    // sum, :142-150) on the un-normalised vector, so the returned ranks carry the same rounding as
    // the reference's; beyond that its fp32 sum is meaningless (0.25 at n = 2^26, SURVEY F7) and the
    // f64 device normalisation is used.
    const bool literal_normalisation = n <= (1 << 24);
    const int rc = pagerank_device(adj_matrix, config, d_ranks, &iters, &residual, &conv, nullptr,
                                   !literal_normalisation, nullptr, 0, d_pvec);
    cudaFree(d_pvec);
    if (rc != 0 && iters == 0) {  // what the reference returns when its first SpMV fails (:105-107, :135-150)
        cudaFree(d_ranks);
        const float init = 1.0f / n;
        for (int i = 0; i < n; ++i) result.ranks[i] = init;
        normalise_literally();
        return 0;
    }
    cudaError_t e = cudaMemcpy(result.ranks, d_ranks, sizeof(float) * n, cudaMemcpyDeviceToHost);
    cudaFree(d_ranks);
    if (e != cudaSuccess) throw CudaException(e);
    if (literal_normalisation) normalise_literally();
    result.iterations = iters;
    result.final_residual = residual;
    result.converged = conv;
    return 0;
}

}  // namespace b200

// -------------------------------------------------------------------- pagerank --
PageRankResult pagerank(const CSRMatrix* adj_matrix, const PageRankConfig* config) {
    PageRankResult result;
    b200::pagerank_to_host(adj_matrix, config, nullptr, &result);
    return result;
}

}  // namespace spmv
