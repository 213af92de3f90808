/*
 * spmv_b200_ppr.h -- C ABI of libspmv_b200_ppr.so: batched personalized PageRank.
 *
 * k personalized PageRank vectors of one graph advance in one loop: every pass over the matrix
 * serves 8 of them, whose ranks are stored node-major (r[node][0..8), 32 bytes per node), so one
 * gathered sector carries the values of all 8 (DESIGN.md section 10).  Link with -lspmv_b200_ppr;
 * the library depends on libspmv_b200.so (same directory) and uses only its C ABI (spmv_b200.h).
 * Conventions as in spmv_b200.h: 0 or a negative spmv_b200_status, nothing throws.
 */
#ifndef SPMV_B200_PPR_H
#define SPMV_B200_PPR_H

#include "spmv_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * k personalized PageRank vectors of one graph in one loop.  Vector c is given sparsely:
 * nodes[offsets[c] .. offsets[c+1]) strictly ascending in [0, n), weights likewise (NULL: all 1).
 * d_ranks: device, n * k floats, node-major (d_ranks[(size_t)i * k + c]).
 * iterations / final_residual / converged: host arrays of k.
 * l2_history: optional host [k][history_capacity].
 *
 * Column c is what spmv_b200_pagerank_device_personalized computes for the dense vector with the
 * same entries: v = w / sum(w) (f64 sum in index order, each entry rounded to fp32), r_0 = 1/n,
 *     r_new[i] = (d * (A r_old)[i] + (d * D_c) * v[i]) + (1 - d) * v[i],   D_c = dangling mass of r_old,
 * stop when the L2 norm of the delta is below the tolerance (checked after every iteration), final
 * f64 normalisation.  Each column stops on its own: from the iteration after it converged on, its
 * vector is carried through unchanged, so iterations[c], final_residual[c], converged[c] and
 * l2_history[c][0 .. iterations[c]) are those of that column alone (entries beyond are untouched).
 * A column's result does not depend on k or on its position in the batch (bit for bit).
 *
 * INVALID_ARGUMENT, before any device work: NULL adj / offsets / d_ranks / result arrays, k <= 0,
 * offsets[0] != 0 or decreasing, nodes NULL with entries, a node out of [0, n), repeated or out of
 * order, a NaN, +-Inf or negative weight, a column whose weights sum to 0 (an empty column too;
 * so every call on n = 0), history_capacity < 0 or > 0 with l2_history NULL.
 * INVALID_DIMENSION for a non-square adjacency (results zeroed, d_ranks untouched); CUDA_MALLOC
 * when the 3 * n * 32 bytes of chunk vectors (plus the plan) do not fit.
 */
SPMV_B200_API int spmv_b200_pagerank_personalized_batch(const spmv_b200_csr* adj,
                                                        const spmv_b200_pagerank_config* config, int k,
                                                        const int* offsets, const int* nodes,
                                                        const float* weights, float* d_ranks, int* iterations,
                                                        float* final_residual, bool* converged,
                                                        float* l2_history, int history_capacity);

/* number of kernels this library (not libspmv_b200.so) has launched in this process so far */
SPMV_B200_API unsigned long long spmv_b200_ppr_launch_count(void);

#ifdef __cplusplus
} /* extern "C" */
#endif

#endif /* SPMV_B200_PPR_H */
