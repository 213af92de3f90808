// pagerank_dist.hpp -- row-sharded PageRank over the GPUs of one box (internal; the C ABI is in
// include/spmv_b200.h, section "multi-GPU").
#pragma once

#include "comm.hpp"
#include "spmv_b200/api.hpp"

#include <cuda_runtime.h>

namespace spmv {
namespace b200 {

// how the rank slices travel between the GPUs
constexpr int kExchangeAuto = -1;       // multicast if the box has NVLS, else peer stores, else NCCL
constexpr int kExchangeNccl = 0;        // ncclBroadcast group + ncclAllGather of the partial sums
constexpr int kExchangeP2P = 1;         // unicast peer stores from inside the step kernel
constexpr int kExchangeMulticast = 2;   // one multimem.st per value through the NVSwitch

struct PrDistResult {
    int iterations = 0;            // as PageRankResult (reference include/spmv/pagerank.h:18-26)
    float final_residual = 0.0f;
    int converged = 0;
    double l1_residual = 0.0;
    int iterations_launched = 0;   // includes the speculative one after convergence
    double device_seconds = 0.0;   // CUDA events around the loop on this rank's stream
    double wall_seconds = 0.0;
    int exchange = 0;              // transport actually used
    int graph_replay = 0;
    int kernels_per_iteration = 0;
};

struct PrDist;
bool nccl_available();
// collective over comm (every rank calls it with its own shard); the shard's device arrays are
// borrowed.  exchange: one of kExchange*.
int pr_dist_create(Comm* comm, const CSRMatrix* shard, int row_offset, int n_global, int exchange, PrDist** out);
void pr_dist_destroy(PrDist* d);  // collective
// collective; fixed_iterations > 0 runs exactly that many iterations (no stop rule)
int pr_dist_run(PrDist* d, const PageRankConfig* config, int fixed_iterations, PrDistResult* out);
// collective; personalized PageRank from the next run on: v_host is the FULL host vector (n_global entries, the
// same on every rank), validated and normalised as pr_personalization_normalise does; this rank keeps its rows.
// nullptr returns to global PageRank.  Drops the cached iteration graphs.
int pr_dist_set_personalization(PrDist* d, const float* v_host);
int pr_dist_exchange(const PrDist* d);
const float* pr_dist_ranks(const PrDist* d);  // device, full length, normalised; valid after a run
cudaStream_t pr_dist_stream(const PrDist* d);
int pr_dist_hub_columns(const PrDist* d);

// One process, n_gpus devices: adj is a HOST CSR; cuts nnz-balanced row shards (work(row) = nnz +
// row_weight), uploads one per device and runs the loop with one host thread per device.
// personalization: host [num_rows] or nullptr (pr_dist_set_personalization).
int pagerank_multi(const CSRMatrix* adj, const PageRankConfig* config, int n_gpus, const int* devices, int exchange,
                   int row_weight, int fixed_iterations, float* ranks_out, PrDistResult* out,
                   const float* personalization = nullptr);

}  // namespace b200
}  // namespace spmv
