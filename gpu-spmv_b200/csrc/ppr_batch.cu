// ppr_batch.cu -- batched personalized PageRank (libspmv_b200_ppr.so): the chunk loop of ppr_core.cuh, with
// each chunk's final vectors normalised into the caller's dense node-major [n][k] ranks.
#include "ppr_core.cuh"
#include "spmv_b200_ppr.h"

namespace spmv {
namespace b200 {
namespace ppr {

// out[i * k + c0 + c] = r[i][c] / (float)sum_c for the `width` lanes of the chunk (as spmv_b200_pr_normalize)
__global__ void __launch_bounds__(256) ppr_scale_kernel(const float* __restrict__ r, long long n, const double* __restrict__ block_sums,
                                                        int blocks, int width, int k, int c0, float* __restrict__ out) {
    __shared__ float s_total[kW];
    if (threadIdx.x < kW) s_total[threadIdx.x] = lane_total(block_sums, blocks, threadIdx.x);
    __syncthreads();
    const long long total = n * width;
    for (long long e = blockIdx.x * 256LL + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * 256) {
        const long long i = e / width;
        const int c = static_cast<int>(e - i * width);
        out[i * k + c0 + c] = normalised(r[i * kW + c], s_total[c]);
    }
}

int run_batch(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, int k, const int* offsets,
              const int* nodes, const float* weights, float* d_ranks, int* iterations, float* final_residual,
              bool* converged, float* l2_history, int history_capacity) {
    if (!d_ranks) return SPMV_B200_INVALID_ARGUMENT;
    const long long n = adj ? adj->num_rows : 0;
    return run_chunks(adj, config, k, offsets, nodes, weights, iterations, final_residual, converged, l2_history,
                      history_capacity,
                      [&](const float* fin, const double* block_sums, int blocks, int c0, int width, cudaStream_t stream) {
                          ppr_scale_kernel<<<grid_for(n * width, 256, kNormBlocksMax), 256, 0, stream>>>(
                              fin, n, block_sums, blocks, width, k, c0, d_ranks);
                          counted(1);
                          return 0;
                      });
}

}  // namespace ppr
}  // namespace b200
}  // namespace spmv

extern "C" {

int spmv_b200_pagerank_personalized_batch(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, int k,
                                          const int* offsets, const int* nodes, const float* weights, float* d_ranks,
                                          int* iterations, float* final_residual, bool* converged, float* l2_history,
                                          int history_capacity) {
    try {
        return spmv::b200::ppr::run_batch(adj, config, k, offsets, nodes, weights, d_ranks, iterations, final_residual,
                                          converged, l2_history, history_capacity);
    } catch (...) {
        return SPMV_B200_OUT_OF_MEMORY;
    }
}

unsigned long long spmv_b200_ppr_launch_count(void) { return spmv::b200::ppr::g_launches.load(); }

}  // extern "C"
