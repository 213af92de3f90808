/*
 * pagerank_personalized_oracle.c -- CPU restatement of personalized PageRank, the checker of
 * tests/test_gpu_pagerank_personalized.py (test infrastructure; the test compiles it on first use with
 * gcc -O2 -ffp-contract=off, the flags of oracle/spmv_oracle.c: no FMA contraction, every fp32 operation
 * rounded on its own).
 *
 * Same structure as orc_pagerank_f64 of oracle/spmv_oracle.c, whose dangling rule (a column whose fp32
 * sum in row-major order is 0) is restated here as orc_find_dangling is.
 */
#include <math.h>
#include <stdlib.h>

#define ORC_API __attribute__((visibility("default")))

/* flags[c] = 1 when column c sums to 0.0f (fp32, row-major order) */
static void find_dangling(int rows, int cols, const float *values, const int *col_indices, const int *row_ptrs,
                          unsigned char *flags)
{
    float *sums = (float *)calloc((size_t)(cols > 0 ? cols : 1), sizeof(float));
    for (int r = 0; r < rows; r++)
        for (int j = row_ptrs[r]; j < row_ptrs[r + 1]; j++) {
            int c = col_indices[j];
            if (c >= 0 && c < cols) sums[c] += values[j];
        }
    for (int c = 0; c < cols; c++) flags[c] = (sums[c] == 0.0f);
    free(sums);
}

/*
 * Personalized PageRank, restated like orc_pagerank_f64 (f64 accumulators,
 * fp32 storage, same stop rule, fixed_iterations, final normalisation).
 * pvec [n] is the caller's personalization vector: normalised here as
 * vhat[i] = (float)((double)pvec[i] / S), S = f64 sum in index order, and
 * the update is r[i] = ((d*y) + (d*D)*vhat[i]) + (1-d)*vhat[i] in fp32,
 * each operation rounded separately.  Returns -1 (nothing written) when an
 * entry is NaN, +-Inf or negative or when S == 0.
 */
ORC_API int orc_pagerank_personalized_f64(int n, int cols, const float *values, const int *col_indices,
                                          const int *row_ptrs, const float *pvec, float damping,
                                          float tolerance, int max_iterations, int fixed_iterations,
                                          float *ranks, double *residual_l2, double *residual_l1,
                                          int *converged)
{
    double S = 0.0;
    for (int i = 0; i < n; i++) {
        if (!isfinite(pvec[i]) || pvec[i] < 0.0f) return -1;
        S += (double)pvec[i];
    }
    if (S == 0.0) return -1;
    float *vhat = (float *)malloc((size_t)(n > 0 ? n : 1) * sizeof(float));
    for (int i = 0; i < n; i++) vhat[i] = (float)((double)pvec[i] / S);
    float *r_old = (float *)malloc((size_t)(n > 0 ? n : 1) * sizeof(float));
    float *r_new = (float *)malloc((size_t)(n > 0 ? n : 1) * sizeof(float));
    unsigned char *dang = (unsigned char *)calloc((size_t)(cols > 0 ? cols : 1), 1);
    float init = 1.0f / n;
    for (int i = 0; i < n; i++) r_old[i] = init;
    float teleport = 1.0f - damping;
    find_dangling(n, cols, values, col_indices, row_ptrs, dang);
    int iters = 0, conv = 0, from_new = 0;
    double l2 = 0.0, l1 = 0.0;
    int limit = fixed_iterations > 0 ? fixed_iterations : max_iterations;
    for (int it = 0; it < limit; it++) {
        double dsum = 0.0;
        for (int c = 0; c < cols; c++)
            if (dang[c] && c < n) dsum += (double)r_old[c];
        float dd = damping * (float)dsum;
        double s2 = 0.0, s1 = 0.0;
        for (int i = 0; i < n; i++) {
            double acc = 0.0;
            for (int j = row_ptrs[i]; j < row_ptrs[i + 1]; j++)
                acc += (double)values[j] * (double)r_old[col_indices[j]];
            float y = (float)acc;
            float v = damping * y + dd * vhat[i] + teleport * vhat[i];
            r_new[i] = v;
            double d = (double)v - (double)r_old[i];
            s2 += d * d;
            s1 += fabs(d);
        }
        l2 = sqrt(s2);
        l1 = s1;
        iters = it + 1;
        if (fixed_iterations <= 0 && (float)l2 < tolerance) { conv = 1; from_new = 1; break; }
        if (fixed_iterations > 0 && it + 1 == limit) { from_new = 1; conv = ((float)l2 < tolerance); break; }
        float *t = r_old; r_old = r_new; r_new = t;
    }
    const float *fin = from_new ? r_new : r_old;
    double sum = 0.0;
    for (int i = 0; i < n; i++) sum += (double)fin[i];
    float sum_f = (float)sum;
    for (int i = 0; i < n; i++) ranks[i] = (sum_f > 0.0f) ? fin[i] / sum_f : fin[i];
    *residual_l2 = l2;
    *residual_l1 = l1;
    *converged = conv;
    free(vhat); free(r_old); free(r_new); free(dang);
    return iters;
}
