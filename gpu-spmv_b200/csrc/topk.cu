// topk.cu -- device-side top-k of a rank vector that is already in HBM.
//
// The reference's pagerank_top_k (src/pagerank.cu:162-185) copies all n (id, rank) pairs into a
// host vector and partial_sorts it: at n = 2^26 that is a 268 MB download plus a 537 MB
// temporary for k results (SURVEY a10, 8f rank 4).  Here the vector stays on the device:
//   1. radix select of the k-th largest value: 4 passes of a 256-bin histogram over an
//      order-preserving uint32 image of the floats (the histogram of each pass is read by
//      the host: 1 KB);
//   2. every element above the threshold is appended to the result (fewer than k);
//   3. elements EQUAL to the threshold fill the remaining places in ascending id order
//      (per-chunk counts -> prefix -> ordered write), so the result is deterministic;
//   4. the k pairs are downloaded and ordered on the host: rank descending, id ascending.
// "identical top-k up to ties" (north_star): values are exactly those of pagerank_top_k;
// among equal ranks the reference's order is unspecified (std::partial_sort), ours is by id.
#include "device_utils.cuh"
#include "internal.hpp"

#include <algorithm>
#include <cub/block/block_scan.cuh>
#include <vector>

namespace spmv {
namespace b200 {
namespace {

constexpr int kBlock = 256;
constexpr int kPerThread = 16;
constexpr int kChunk = kBlock * kPerThread;  // elements per CTA in the ordered passes

using dev::order_key;

// histogram of byte `shift / 8` of the keys whose higher bytes equal `prefix`
__global__ void __launch_bounds__(kBlock)
topk_hist_kernel(const float* __restrict__ v, int n, unsigned prefix, unsigned prefix_mask, int shift,
                 unsigned* __restrict__ hist) {
    __shared__ unsigned s_hist[256];
    s_hist[threadIdx.x] = 0;
    __syncthreads();
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kBlock) {
        const unsigned key = order_key(v[i]);
        if ((key & prefix_mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (s_hist[threadIdx.x]) atomicAdd(hist + threadIdx.x, s_hist[threadIdx.x]);
}

__global__ void __launch_bounds__(kBlock)
topk_gather_greater_kernel(const float* __restrict__ v, int n, unsigned threshold, int* __restrict__ out_ids,
                           float* __restrict__ out_vals, int* __restrict__ counter) {
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kBlock) {
        const float x = v[i];
        if (order_key(x) > threshold) {
            const int at = atomicAdd(counter, 1);
            out_ids[at] = static_cast<int>(i);
            out_vals[at] = x;
        }
    }
}

__global__ void __launch_bounds__(kBlock)
topk_tie_count_kernel(const float* __restrict__ v, int n, unsigned threshold, int* __restrict__ chunk_count) {
    __shared__ int s_total;
    if (threadIdx.x == 0) s_total = 0;
    __syncthreads();
    const long long base = static_cast<long long>(blockIdx.x) * kChunk + static_cast<long long>(threadIdx.x) * kPerThread;
    int c = 0;
    for (int k = 0; k < kPerThread; ++k)
        if (base + k < n && order_key(v[base + k]) == threshold) ++c;
    if (c) atomicAdd(&s_total, c);
    __syncthreads();
    if (threadIdx.x == 0) chunk_count[blockIdx.x] = s_total;
}

// writes the ties whose rank among all ties (ascending id) is below `need`
__global__ void __launch_bounds__(kBlock)
topk_tie_write_kernel(const float* __restrict__ v, int n, unsigned threshold, const int* __restrict__ chunk_start,
                      int need, int out_base, int* __restrict__ out_ids, float* __restrict__ out_vals) {
    using Scan = cub::BlockScan<int, kBlock>;
    __shared__ typename Scan::TempStorage temp;
    const int start = chunk_start[blockIdx.x];
    if (start >= need) return;  // block-uniform
    const long long base = static_cast<long long>(blockIdx.x) * kChunk + static_cast<long long>(threadIdx.x) * kPerThread;
    int c = 0;
    for (int k = 0; k < kPerThread; ++k)
        if (base + k < n && order_key(v[base + k]) == threshold) ++c;
    int before = 0;
    Scan(temp).ExclusiveSum(c, before);
    int at = start + before;
    for (int k = 0; k < kPerThread; ++k) {
        if (base + k < n && order_key(v[base + k]) == threshold) {
            if (at < need) {
                out_ids[out_base + at] = static_cast<int>(base + k);
                out_vals[out_base + at] = v[base + k];
            }
            ++at;
        }
    }
}

}  // namespace

int pagerank_top_k_device(const float* d_ranks, int n, int k, TopKNode* top_k) {
    if (!d_ranks || !top_k || n < 0 || k < 0) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    const int kk = k < n ? k : n;
    if (kk == 0) return 0;
    cudaStream_t stream = nullptr;
    const int chunks = (n + kChunk - 1) / kChunk;
    unsigned* d_hist = nullptr;
    int *d_ids = nullptr, *d_counter = nullptr, *d_chunk = nullptr;
    float* d_vals = nullptr;
    auto cleanup = [&]() { cudaFree(d_hist); cudaFree(d_ids); cudaFree(d_vals); cudaFree(d_counter); cudaFree(d_chunk); };
    auto fail = [&](SpMVError code) {
        cudaGetLastError();
        cleanup();
        return static_cast<int>(code);
    };
    if (cudaMalloc(&d_hist, 256 * sizeof(unsigned)) != cudaSuccess || cudaMalloc(&d_ids, sizeof(int) * kk) != cudaSuccess ||
        cudaMalloc(&d_vals, sizeof(float) * kk) != cudaSuccess || cudaMalloc(&d_counter, sizeof(int)) != cudaSuccess ||
        cudaMalloc(&d_chunk, sizeof(int) * chunks) != cudaSuccess)
        return fail(SpMVError::CUDA_MALLOC);
    const unsigned grid = static_cast<unsigned>(std::min<long long>((static_cast<long long>(n) + kBlock - 1) / kBlock, 148 * 16));

    // 1. radix select: after the loop `prefix` is the key of the kk-th largest element
    unsigned prefix = 0, mask = 0;
    long long above = 0;  // elements known to be larger than every key with this prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
        unsigned h[256];
        cudaMemsetAsync(d_hist, 0, sizeof(h), stream);
        topk_hist_kernel<<<grid, kBlock, 0, stream>>>(d_ranks, n, prefix, mask, shift, d_hist);
        if (cudaMemcpyAsync(h, d_hist, sizeof(h), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
            cudaStreamSynchronize(stream) != cudaSuccess)
            return fail(SpMVError::KERNEL_LAUNCH);
        int bin = 255;
        for (; bin > 0; --bin) {
            if (above + h[bin] >= kk) break;
            above += h[bin];
        }
        prefix |= static_cast<unsigned>(bin) << shift;
        mask |= 255u << shift;
    }
    count_launches(4);
    const int need = kk - static_cast<int>(above);  // places left for elements equal to the threshold (>= 1)

    // 2. everything above the threshold
    cudaMemsetAsync(d_counter, 0, sizeof(int), stream);
    topk_gather_greater_kernel<<<grid, kBlock, 0, stream>>>(d_ranks, n, prefix, d_ids, d_vals, d_counter);
    // 3. ties, lowest ids first
    topk_tie_count_kernel<<<chunks, kBlock, 0, stream>>>(d_ranks, n, prefix, d_chunk);
    std::vector<int> counts(static_cast<size_t>(chunks));
    if (cudaMemcpyAsync(counts.data(), d_chunk, sizeof(int) * chunks, cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
        cudaStreamSynchronize(stream) != cudaSuccess)
        return fail(SpMVError::KERNEL_LAUNCH);
    int run = 0;
    for (int c = 0; c < chunks; ++c) {
        const int here = counts[static_cast<size_t>(c)];
        counts[static_cast<size_t>(c)] = run;
        run = run > need ? run : run + here;  // saturates: later chunks are not needed
    }
    cudaMemcpyAsync(d_chunk, counts.data(), sizeof(int) * chunks, cudaMemcpyHostToDevice, stream);
    topk_tie_write_kernel<<<chunks, kBlock, 0, stream>>>(d_ranks, n, prefix, d_chunk, need, static_cast<int>(above), d_ids,
                                                         d_vals);
    count_launches(3);
    // 4. download and order: rank descending, id ascending
    std::vector<int> ids(static_cast<size_t>(kk));
    std::vector<float> vals(static_cast<size_t>(kk));
    if (cudaMemcpyAsync(ids.data(), d_ids, sizeof(int) * kk, cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
        cudaMemcpyAsync(vals.data(), d_vals, sizeof(float) * kk, cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
        cudaStreamSynchronize(stream) != cudaSuccess || cudaGetLastError() != cudaSuccess)
        return fail(SpMVError::KERNEL_LAUNCH);
    cleanup();
    std::vector<int> order(static_cast<size_t>(kk));
    for (int i = 0; i < kk; ++i) order[static_cast<size_t>(i)] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        const float va = vals[static_cast<size_t>(a)], vb = vals[static_cast<size_t>(b)];
        if (va != vb) return va > vb;
        return ids[static_cast<size_t>(a)] < ids[static_cast<size_t>(b)];
    });
    for (int i = 0; i < kk; ++i) {
        top_k[i].node_id = ids[static_cast<size_t>(order[static_cast<size_t>(i)])];
        top_k[i].rank = vals[static_cast<size_t>(order[static_cast<size_t>(i)])];
    }
    return 0;
}

}  // namespace b200
}  // namespace spmv
