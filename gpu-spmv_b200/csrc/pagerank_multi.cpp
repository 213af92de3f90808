// pagerank_multi.cpp -- PageRank over n_gpus devices from ONE process: the multi-GPU member of the
// reference's signature family pagerank(adj, config) -> ranks (reference include/spmv/pagerank.h:29-32,
// src/pagerank.cu:50-153), for a C / C++ caller that has a host CSR and a box of GPUs and no launcher.
// Rows are cut into contiguous shards that balance work(row) = nnz + row_weight, one host thread per
// device uploads its shard and runs the same per-rank loop as the one-process-per-GPU form
// (pagerank_dist.cu), the ranks meeting through a ThreadComm instead of sockets.
#include "pagerank_dist.hpp"

#include "internal.hpp"

#include <atomic>
#include <thread>
#include <vector>

extern "C" int spmv_b200_partition_rows_weighted(const int* row_ptrs, int num_rows, int parts, int row_weight, int* bounds);

namespace spmv {
namespace b200 {

int pagerank_multi(const CSRMatrix* adj, const PageRankConfig* config, int n_gpus, const int* devices, int exchange,
                   int row_weight, int fixed_iterations, float* ranks_out, PrDistResult* out,
                   const float* personalization) {
    if (!adj || !ranks_out || n_gpus < 1 || n_gpus > 8) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (personalization) {  // rejected before any device work (every rank checks it again)
        std::vector<float> vhat;
        const int rc = pr_personalization_normalise(personalization, adj->num_rows, &vhat);
        if (rc != 0) return rc;
    }
    if (!adj->row_ptrs || (adj->nnz > 0 && (!adj->col_indices || !adj->values)))
        return static_cast<int>(SpMVError::INVALID_FORMAT);  // host arrays are what gets sharded
    if (adj->num_cols != adj->num_rows) return static_cast<int>(SpMVError::INVALID_DIMENSION);
    // devices == NULL: ranks 0 .. n_gpus-1 on devices 0 .. n_gpus-1.  An explicit list may name a device
    // more than once (several ranks share a GPU: the peer-store exchange and the flag barrier work
    // between streams of one device exactly as between devices -- how the sharded path is tested on a
    // one-GPU box; the multicast and NCCL transports need distinct devices).
    int visible = 0;
    bool devices_ok = cudaGetDeviceCount(&visible) == cudaSuccess && (devices || visible >= n_gpus);
    for (int r = 0; devices_ok && devices && r < n_gpus; ++r) devices_ok = devices[r] >= 0 && devices[r] < visible;
    if (!devices_ok) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    }
    const int n = adj->num_rows;
    std::vector<int> bounds(n_gpus + 1, 0);
    if (spmv_b200_partition_rows_weighted(adj->row_ptrs, n, n_gpus, row_weight < 0 ? 0 : row_weight, bounds.data()) != 0)
        return static_cast<int>(SpMVError::INVALID_ARGUMENT);

    ThreadCommGroup* group = thread_comm_group_create(n_gpus);
    std::vector<int> rcs(n_gpus, 0);
    std::vector<PrDistResult> results(n_gpus);
    auto worker = [&](int rank) {
        Comm* comm = thread_comm_get(group, rank);
        int rc = 0;
        if (cudaSetDevice(devices ? devices[rank] : rank) != cudaSuccess) rc = static_cast<int>(SpMVError::INVALID_ARGUMENT);
        // the shard: rows [lo, hi), row_ptrs rebased to 0, global column ids; values / columns alias the parent
        const int lo = bounds[rank], hi = bounds[rank + 1];
        const int base = adj->row_ptrs[lo];
        std::vector<int> rp(static_cast<size_t>(hi - lo) + 1);
        for (int i = lo; i <= hi; ++i) rp[i - lo] = adj->row_ptrs[i] - base;
        CSRMatrix shard{};
        shard.num_rows = hi - lo;
        shard.num_cols = n;
        shard.nnz = adj->row_ptrs[hi] - base;
        shard.row_ptrs = rp.data();
        shard.col_indices = shard.nnz > 0 ? adj->col_indices + base : nullptr;
        shard.values = shard.nnz > 0 ? adj->values + base : nullptr;
        shard.owns_host_memory = false;
        if (rc == 0) rc = csr_to_gpu(&shard);
        if (rc == 0 && shard.nnz == 0 && !shard.d_col_indices) {  // an empty shard still needs non-null device arrays
            if (cudaMalloc(&shard.d_col_indices, 16) != cudaSuccess || cudaMalloc(&shard.d_values, 16) != cudaSuccess) rc = static_cast<int>(SpMVError::CUDA_MALLOC);
        }
        // every rank must reach the collectives, also after a local failure: agree first
        int ok = rc == 0 ? 1 : 0;
        std::vector<int> all(n_gpus, 0);
        comm->allgather(&ok, all.data(), sizeof(int));
        bool everyone = true;
        for (int v : all) everyone = everyone && v != 0;
        PrDist* d = nullptr;
        if (everyone) {
            rc = pr_dist_create(comm, &shard, lo, n, exchange, &d);
            if (rc == 0) {
                if (personalization) rc = pr_dist_set_personalization(d, personalization);
                if (rc == 0) rc = pr_dist_run(d, config, fixed_iterations, &results[rank]);
                if (rc == 0 && rank == 0 &&
                    cudaMemcpy(ranks_out, pr_dist_ranks(d), sizeof(float) * static_cast<size_t>(n), cudaMemcpyDeviceToHost) != cudaSuccess) {
                    cudaGetLastError();
                    rc = static_cast<int>(SpMVError::CUDA_MEMCPY);
                }
                pr_dist_destroy(d);
            }
        } else if (rc == 0) {
            rc = static_cast<int>(SpMVError::CUDA_MALLOC);
        }
        csr_free_gpu(&shard);
        rcs[rank] = rc;
    };
    std::vector<std::thread> threads;
    for (int r = 1; r < n_gpus; ++r) threads.emplace_back(worker, r);
    int caller_device = 0;
    cudaGetDevice(&caller_device);
    worker(0);
    for (auto& t : threads) t.join();
    cudaSetDevice(caller_device);
    thread_comm_group_destroy(group);
    int rc = 0;
    for (int r = 0; r < n_gpus; ++r)
        if (rcs[r] != 0 && rc == 0) rc = rcs[r];
    if (out) {
        *out = results[0];
        for (int r = 1; r < n_gpus; ++r)  // the slowest rank sets the time
            if (results[r].device_seconds > out->device_seconds) out->device_seconds = results[r].device_seconds;
    }
    return rc;
}

}  // namespace b200
}  // namespace spmv
