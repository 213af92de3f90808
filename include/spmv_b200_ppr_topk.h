/*
 * spmv_b200_ppr_topk.h -- C ABI of libspmv_b200_ppr_topk.so: per-seed top-K personalized PageRank.
 *
 * The loop of spmv_b200_pagerank_personalized_batch (spmv_b200_ppr.h), but each column's result is
 * its `top` largest ranks instead of a dense [n][k] matrix: device memory depends on n and on
 * k * top, never on n * k, so thousands of seeds fit where the dense output would not (DESIGN.md
 * section 11).  Link with -lspmv_b200_ppr_topk; the library depends on libspmv_b200.so (same
 * directory) and uses only its C ABI (spmv_b200.h).
 * Conventions as in spmv_b200.h: 0 or a negative spmv_b200_status, nothing throws.
 */
#ifndef SPMV_B200_PPR_TOPK_H
#define SPMV_B200_PPR_TOPK_H

#include "spmv_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * k personalized PageRank vectors of one graph, each reduced to its `top` best nodes.
 * adj, config, k, offsets, nodes, weights, iterations, final_residual, converged, l2_history and
 * history_capacity: exactly as spmv_b200_pagerank_personalized_batch, and the four results are bit for
 * bit what it returns for the same inputs.
 * d_ids, d_vals: device, k * top each, row-major (row c at (size_t)c * top).  Row c holds the min(top, n)
 * largest entries of column c of the batch's d_ranks, with the same fp32 bits, ordered by rank
 * descending, then node id ascending among equal ranks (the order of spmv_b200_pagerank_top_k_device;
 * -0 and +0 are equal); places [n, top) hold id -1 and value 0.0f.
 *
 * INVALID_ARGUMENT, before any device work: every rejection of the batch (d_ranks aside), top < 1 or
 * top > 1024, d_ids or d_vals NULL.  INVALID_DIMENSION for a non-square adjacency (results zeroed,
 * d_ids / d_vals untouched).  CUDA_MALLOC when the batch's working set (3 * n * 32 bytes plus the plan)
 * and the selection's 8 * ceil(n / 4096) + 2048 words do not fit.
 */
SPMV_B200_API int spmv_b200_pagerank_personalized_batch_top_k(const spmv_b200_csr* adj,
                                                              const spmv_b200_pagerank_config* config, int k,
                                                              const int* offsets, const int* nodes,
                                                              const float* weights, int top, int* d_ids,
                                                              float* d_vals, int* iterations,
                                                              float* final_residual, bool* converged,
                                                              float* l2_history, int history_capacity);

/* number of kernels this library (not libspmv_b200.so) has launched in this process so far */
SPMV_B200_API unsigned long long spmv_b200_ppr_topk_launch_count(void);

#ifdef __cplusplus
} /* extern "C" */
#endif

#endif /* SPMV_B200_PPR_TOPK_H */
