// aux_kernels.cu -- small device kernels around the hot path: PageRank set-up
// (column sums, dangling bitmask, initial vector, normalisation) and the
// device-side ELL assembly.  None of them is on the per-iteration critical
// path except next_dsum (one thread).
#include "device_utils.cuh"
#include "internal.hpp"

namespace spmv {
namespace b200 {
namespace {

constexpr int kBlock = 256;

inline unsigned grid_for(long long n, int per_block = kBlock, unsigned cap = 148u * 16u) {
    long long b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return static_cast<unsigned>(b < cap ? b : cap);
}
static_assert(kPrScratchDoubles >= 148 * 16, "pr_init and normalize store one double per CTA of grid_for's grid");

// d_colsum[c] += values[j] for every stored entry (find_dangling_nodes, reference
// src/pagerank.cu:30-40).  The sums are accumulated in f64: an fp32 value enters an f64 sum without
// rounding as long as the column's partial sums fit 53 bits, which holds for every column of a
// column-normalised adjacency matrix (k copies of 1/k) and for any column whose entries span
// less than 2^29 in magnitude -- and a sum that is never rounded does not depend on the order of
// the atomics.  So the set of dangling nodes (sum == 0) is deterministic, and it is the TRUE
// cancellation set; the reference's sequential fp32 sum can differ from it only for mixed-sign
// columns whose fp32 partial sums round (documented in DESIGN.md section 5).
__global__ void colsum_kernel(int nnz, int cols, const int* __restrict__ col_indices,
                              const float* __restrict__ values, double* __restrict__ colsum) {
    for (long long j = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; j < nnz;
         j += static_cast<long long>(gridDim.x) * kBlock) {
        const int c = dev::ld_stream_i(col_indices + j);
        if (c >= 0 && c < cols) atomicAdd(colsum + c, static_cast<double>(dev::ld_stream_f(values + j)));
    }
}

// bit c = (colsum[c] == 0), reference src/pagerank.cu:42-46
// (nodes at or beyond valid_cols have no column and are never dangling)
__global__ void dangling_bits_kernel(const double* __restrict__ colsum, int n, int valid_cols,
                                     uint32_t* __restrict__ bits) {
    const int words = (n + 31) / 32;
    for (int w = blockIdx.x * kBlock + threadIdx.x; w < words; w += gridDim.x * kBlock) {
        uint32_t m = 0;
        const int lim = min(32, n - w * 32);
        for (int b = 0; b < lim; ++b) {
            const int c = w * 32 + b;
            m |= ((c < valid_cols && static_cast<float>(colsum[c]) == 0.0f) ? 1u : 0u) << b;
        }
        bits[w] = m;
    }
}

// r[i] = 1/n (reference src/pagerank.cu:69-72); counts dangling nodes per CTA
__global__ void pr_init_kernel(int n, float init, const uint32_t* __restrict__ bits, float* __restrict__ r,
                               double* __restrict__ block_counts) {
    __shared__ unsigned s[kBlock / 32];
    unsigned cnt = 0;
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kBlock) {
        r[i] = init;
        cnt += (bits[i >> 5] >> (i & 31)) & 1u;
    }
    cnt = dev::warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int w = 0; w < kBlock / 32; ++w) t += s[w];
        block_counts[blockIdx.x] = static_cast<double>(t);
    }
}

// dsum = (float)(count * init): the dangling mass of the uniform start vector
__global__ void pr_init_finish_kernel(const double* __restrict__ block_counts, int blocks, float init,
                                      float* __restrict__ dsum) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < blocks; ++b) t += block_counts[b];
        *dsum = static_cast<float>(t * static_cast<double>(init));
    }
}

__global__ void next_dsum_kernel(const double* __restrict__ partial, float* __restrict__ dsum) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *dsum = static_cast<float>(partial[2]);
}

// per-CTA f64 sums of r
__global__ void sum_kernel(const float* __restrict__ r, int n, double* __restrict__ block_sums) {
    __shared__ double s[kBlock / 32];
    double acc = 0.0;
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kBlock)
        acc += static_cast<double>(r[i]);
    acc = dev::warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kBlock / 32; ++w) t += s[w];
        block_sums[blockIdx.x] = t;
    }
}

// out[i] = r[i] / (float)sum when sum > 0 (reference src/pagerank.cu:142-150)
__global__ void scale_kernel(const float* __restrict__ r, int n, const double* __restrict__ block_sums,
                             int blocks, float* __restrict__ out) {
    __shared__ float s_total;
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < blocks; ++b) t += block_sums[b];
        s_total = static_cast<float>(t);
    }
    __syncthreads();
    const float total = s_total;
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kBlock)
        out[i] = total > 0.0f ? __fdiv_rn(r[i], total) : r[i];
}

// ell_from_csr on the device (reference src/ell_matrix.cpp:139-156): thread per
// row; slot k of row i at k*rows + i; unused slots col -1 / value 0.
__global__ void ell_from_csr_kernel(int rows, int width, const int* __restrict__ row_ptrs,
                                    const int* __restrict__ col_indices, const float* __restrict__ values,
                                    float* __restrict__ ell_values, int* __restrict__ ell_cols) {
    const int i = blockIdx.x * kBlock + threadIdx.x;
    if (i >= rows) return;
    const int a = row_ptrs[i], b = row_ptrs[i + 1];
    for (int k = 0; k < width; ++k) {
        const size_t slot = static_cast<size_t>(k) * rows + i;
        const int j = a + k;
        ell_values[slot] = j < b ? values[j] : 0.0f;
        ell_cols[slot] = j < b ? col_indices[j] : -1;
    }
}

__global__ void max_row_len_kernel(int rows, const int* __restrict__ row_ptrs, int* __restrict__ out) {
    int m = 0;
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < rows;
         i += static_cast<long long>(gridDim.x) * kBlock)
        m = max(m, row_ptrs[i + 1] - row_ptrs[i]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

}  // namespace

cudaError_t launch_colsum(const CsrView& A, double* d_colsum, cudaStream_t stream) {
    if (A.nnz <= 0) return cudaSuccess;
    colsum_kernel<<<grid_for(A.nnz), kBlock, 0, stream>>>(A.nnz, A.cols, A.col_indices, A.values, d_colsum);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_dangling_bits(const double* d_colsum, int n, int valid_cols, uint32_t* d_bits,
                                 cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    dangling_bits_kernel<<<grid_for((n + 31) / 32), kBlock, 0, stream>>>(d_colsum, n, valid_cols, d_bits);
    count_launches(1);
    return cudaGetLastError();
}

// d_tmp: kPrScratchDoubles doubles
cudaError_t launch_pr_init(int n, const uint32_t* d_bits, float* d_r, float* d_dsum, double* d_tmp,
                           cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const float init = 1.0f / n;
    const unsigned blocks = grid_for(n);
    pr_init_kernel<<<blocks, kBlock, 0, stream>>>(n, init, d_bits, d_r, d_tmp);
    pr_init_finish_kernel<<<1, 32, 0, stream>>>(d_tmp, static_cast<int>(blocks), init, d_dsum);
    count_launches(2);
    return cudaGetLastError();
}

cudaError_t launch_next_dsum(const double* d_partial, float* d_dsum, cudaStream_t stream) {
    next_dsum_kernel<<<1, 32, 0, stream>>>(d_partial, d_dsum);
    count_launches(1);
    return cudaGetLastError();
}

// d_tmp: kPrScratchDoubles doubles
cudaError_t launch_normalize(const float* d_r, int n, float* d_out, double* d_tmp, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned blocks = grid_for(n);
    sum_kernel<<<blocks, kBlock, 0, stream>>>(d_r, n, d_tmp);
    scale_kernel<<<blocks, kBlock, 0, stream>>>(d_r, n, d_tmp, static_cast<int>(blocks), d_out);
    count_launches(2);
    return cudaGetLastError();
}

cudaError_t launch_ell_from_csr(const CsrView& A, int width, float* ell_values, int* ell_cols,
                                cudaStream_t stream) {
    if (A.rows <= 0 || width <= 0) return cudaSuccess;
    ell_from_csr_kernel<<<(A.rows + kBlock - 1) / kBlock, kBlock, 0, stream>>>(A.rows, width, A.row_ptrs, A.col_indices,
                                                                             A.values, ell_values, ell_cols);
    count_launches(1);
    return cudaGetLastError();
}

// *d_out must be zero on entry
cudaError_t launch_max_row_len(const CsrView& A, int* d_out, cudaStream_t stream) {
    if (A.rows <= 0) return cudaSuccess;
    max_row_len_kernel<<<grid_for(A.rows), kBlock, 0, stream>>>(A.rows, A.row_ptrs, d_out);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace b200
}  // namespace spmv
