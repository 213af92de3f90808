// ppr_topk.cu -- per-seed top-K personalized PageRank (libspmv_b200_ppr_topk.so).
//
// The chunk loop of ppr_core.cuh, finished by a radix select over each chunk's node-major [n][8] final
// vector instead of the dense [n][k] output: device memory depends on n and on k * top, never on n * k.
// Each selected value is normalised(r[i][c], lane_total) -- the same expression ppr_scale_kernel writes --
// so a row holds exactly the bits of the corresponding column of spmv_b200_pagerank_personalized_batch.
// Per chunk, all on the stream (the host waits nowhere the batch does not):
//   ppr_topk_begin_kernel      lane totals from ppr_sum_kernel's per-CTA sums; selection state reset
//   ppr_topk_hist_kernel  x4   256-bin histogram of one key byte per lane (keys whose higher bytes match the
//                              lane's prefix), each node's 32 bytes read once for all 8 lanes
//   ppr_topk_bin_kernel   x4   per lane: the bin holding the kk-th largest key; extends the prefix, counts
//                              the entries above it
//   ppr_topk_above_kernel      appends every entry above the lane's threshold key to its output row and
//                              counts the entries equal to it per block of kTieChunk nodes
//   ppr_topk_tie_scan_kernel   per lane: exclusive prefix of those counts
//   ppr_topk_tie_write_kernel  ties fill the row's remaining places in ascending node order
//   ppr_topk_sort_kernel       one CTA per lane sorts its kk entries by (key descending, node ascending) and
//                              pads places [kk, top) with (-1, 0.0f): the row does not depend on atomics' order
// The key is dev::order_key, as in spmv_b200_pagerank_top_k_device (-0 equals +0).
#include "ppr_core.cuh"
#include "spmv_b200_ppr_topk.h"

#include <cub/block/block_scan.cuh>

namespace spmv {
namespace b200 {
namespace ppr {

constexpr int kTopMax = 1024;                   // one CTA sorts a row's entries in shared memory
constexpr int kSel = 256;                       // threads of the selection kernels
constexpr int kTiePer = 16;                     // nodes per thread in the tie passes
constexpr int kTieChunk = kSel * kTiePer;       // nodes per tie-count block
constexpr int kSelBlocksMax = 148 * 8;

// Per-chunk selection state, device-resident; lane c describes column c0 + c.
struct Select {
    float total[kW];      // a rank is normalised(r[i][c], total[c])
    unsigned prefix[kW];  // key bits fixed so far; after the 4 passes the key of the lane's kk-th largest rank
    int above[kW];        // entries whose key is larger than every key with this prefix
    int appended[kW];     // entries above the threshold written to the lane's row so far
};

__device__ __forceinline__ void node_ranks(const float* __restrict__ r, long long i, const float (&t)[kW], float (&v)[kW]) {
    load8(r + i * kW, v);
#pragma unroll
    for (int c = 0; c < kW; ++c) v[c] = normalised(v[c], t[c]);
}

__device__ __forceinline__ void load_select(const Select* sel, float (&t)[kW], unsigned (&key)[kW]) {
#pragma unroll
    for (int c = 0; c < kW; ++c) {
        t[c] = sel->total[c];
        key[c] = sel->prefix[c];
    }
}

__global__ void __launch_bounds__(kSel) ppr_topk_begin_kernel(const double* __restrict__ block_sums, int blocks,
                                                              Select* __restrict__ sel, unsigned* __restrict__ hist) {
    const int c = threadIdx.x;
    if (c < kW) {
        sel->total[c] = lane_total(block_sums, blocks, c);
        sel->prefix[c] = 0;
        sel->above[c] = 0;
        sel->appended[c] = 0;
    }
    for (int j = threadIdx.x; j < kW * 256; j += kSel) hist[j] = 0;
}

// hist[c][b] += number of nodes whose lane-c key has byte `shift / 8` equal to b and higher bytes equal to the prefix
__global__ void __launch_bounds__(kSel)
ppr_topk_hist_kernel(const float* __restrict__ r, long long n, int width, int shift, const Select* __restrict__ sel,
                     unsigned* __restrict__ hist) {
    __shared__ unsigned s_hist[kW * 256];
    for (int j = threadIdx.x; j < kW * 256; j += kSel) s_hist[j] = 0;
    float t[kW];
    unsigned prefix[kW];
    load_select(sel, t, prefix);
    const unsigned mask = shift == 24 ? 0u : ~0u << (shift + 8);
    __syncthreads();
    // block-uniform trip count: every thread of a warp takes part in the match below
    for (long long base = blockIdx.x * static_cast<long long>(kSel); base < n; base += static_cast<long long>(gridDim.x) * kSel) {
        const long long i = base + threadIdx.x;
        float v[kW];
        if (i < n) node_ranks(r, i, t, v);
#pragma unroll
        for (int c = 0; c < kW; ++c) {
            if (c >= width) break;
            const unsigned key = i < n ? dev::order_key(v[c]) : 0u;
            const unsigned bin = (i < n && (key & mask) == prefix[c]) ? (key >> shift) & 255u : 256u;
            // one shared atomic per distinct bin of the warp: ranks crowd into few bins of the high bytes
            const unsigned peers = __match_any_sync(0xffffffffu, bin);
            if (bin < 256u && static_cast<int>(threadIdx.x & 31) == __ffs(peers) - 1)
                atomicAdd(&s_hist[c * 256 + bin], static_cast<unsigned>(__popc(peers)));
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < width * 256; j += kSel)
        if (s_hist[j]) atomicAdd(hist + j, s_hist[j]);
}

// warp c picks lane c's bin: the highest bin b with above + count(bins > b) < kk <= above + count(bins >= b);
// the lane's histogram is cleared for the next pass
__global__ void __launch_bounds__(kW * 32) ppr_topk_bin_kernel(unsigned* __restrict__ hist, int shift, int kk, int width,
                                                               Select* __restrict__ sel) {
    __shared__ unsigned s_h[kW][256];
    const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (c >= width) return;  // warp-uniform
    for (int j = lane; j < 256; j += 32) {
        s_h[c][j] = hist[c * 256 + j];
        hist[c * 256 + j] = 0;
    }
    __syncwarp();
    if (lane == 0) {
        long long above = sel->above[c];
        int bin = 255;
        for (; bin > 0; --bin) {
            if (above + s_h[c][bin] >= kk) break;
            above += s_h[c][bin];
        }
        sel->prefix[c] |= static_cast<unsigned>(bin) << shift;
        sel->above[c] = static_cast<int>(above);
    }
}

// Entries above the threshold go to their row (there are above[c] < kk of them); entries equal to it are counted
// per block: ties[c * gridDim.x + block].  Block b covers nodes [b * kTieChunk, (b + 1) * kTieChunk).
__global__ void __launch_bounds__(kSel)
ppr_topk_above_kernel(const float* __restrict__ r, long long n, int width, Select* __restrict__ sel, int top, int c0,
                      int* __restrict__ ids, float* __restrict__ vals, int* __restrict__ ties) {
    __shared__ int s_ties[kW];
    if (threadIdx.x < kW) s_ties[threadIdx.x] = 0;
    float t[kW];
    unsigned thr[kW];
    load_select(sel, t, thr);
    __syncthreads();
    int cnt[kW];
#pragma unroll
    for (int c = 0; c < kW; ++c) cnt[c] = 0;
    const long long b0 = blockIdx.x * static_cast<long long>(kTieChunk);
    for (int j = 0; j < kTiePer; ++j) {
        const long long i = b0 + j * kSel + threadIdx.x;
        if (i >= n) break;
        float v[kW];
        node_ranks(r, i, t, v);
#pragma unroll
        for (int c = 0; c < kW; ++c) {
            if (c >= width) break;
            const unsigned key = dev::order_key(v[c]);
            if (key > thr[c]) {
                const size_t at = static_cast<size_t>(c0 + c) * top + atomicAdd(&sel->appended[c], 1);
                ids[at] = static_cast<int>(i);
                vals[at] = v[c];
            } else if (key == thr[c]) {
                ++cnt[c];
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kW; ++c) {
        const unsigned s = dev::warp_sum(static_cast<unsigned>(cnt[c]));
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(&s_ties[c], static_cast<int>(s));
    }
    __syncthreads();
    if (threadIdx.x < width) ties[static_cast<size_t>(threadIdx.x) * gridDim.x + blockIdx.x] = s_ties[threadIdx.x];
}

// CTA c: ties[c][b] becomes the number of lane-c ties in blocks before b (at most n: no overflow)
__global__ void __launch_bounds__(kSel) ppr_topk_tie_scan_kernel(int* __restrict__ ties, int blocks) {
    using Scan = cub::BlockScan<int, kSel>;
    __shared__ typename Scan::TempStorage temp;
    int* row = ties + static_cast<size_t>(blockIdx.x) * blocks;
    int run = 0;
    for (int base = 0; base < blocks; base += kSel * kTiePer) {
        int x[kTiePer];
        const int first = base + threadIdx.x * kTiePer;
#pragma unroll
        for (int j = 0; j < kTiePer; ++j) x[j] = first + j < blocks ? row[first + j] : 0;
        int total = 0;
        Scan(temp).ExclusiveSum(x, x, total);
#pragma unroll
        for (int j = 0; j < kTiePer; ++j)
            if (first + j < blocks) row[first + j] = run + x[j];
        run += total;
        __syncthreads();  // temp is reused
    }
}

// The ties whose rank among the lane's ties (ascending node) is below need = kk - above fill the row after the
// entries above the threshold.  Thread t of block b reads nodes b * kTieChunk + t * kTiePer + [0, kTiePer).
__global__ void __launch_bounds__(kSel)
ppr_topk_tie_write_kernel(const float* __restrict__ r, long long n, int width, const Select* __restrict__ sel,
                          const int* __restrict__ ties, int kk, int top, int c0, int* __restrict__ ids,
                          float* __restrict__ vals) {
    using Scan = cub::BlockScan<int, kSel>;
    __shared__ typename Scan::TempStorage temp;
    const long long base = blockIdx.x * static_cast<long long>(kTieChunk) + static_cast<long long>(threadIdx.x) * kTiePer;
    for (int c = 0; c < width; ++c) {
        const int above = sel->above[c];
        const int need = kk - above;
        const int start = ties[static_cast<size_t>(c) * gridDim.x + blockIdx.x];
        if (start >= need) continue;  // block-uniform
        const float t = sel->total[c];
        const unsigned thr = sel->prefix[c];
        unsigned tied = 0;  // bit j: node base + j is a tie
#pragma unroll
        for (int j = 0; j < kTiePer; ++j)
            if (base + j < n && dev::order_key(normalised(r[(base + j) * kW + c], t)) == thr) tied |= 1u << j;
        int before = 0;
        Scan(temp).ExclusiveSum(__popc(tied), before);
        for (int at = start + before; tied && at < need; ++at, tied &= tied - 1) {
            const int j = __ffs(tied) - 1;
            const size_t o = static_cast<size_t>(c0 + c) * top + above + at;
            ids[o] = static_cast<int>(base + j);
            vals[o] = normalised(r[(base + j) * kW + c], t);
        }
        __syncthreads();  // temp is reused by the next lane
    }
}

// CTA c sorts the kk entries of row c0 + c by (key descending, node ascending): each entry's place is the number of
// entries before it (the pairs are distinct).  Places [kk, top) get (-1, 0.0f).
__global__ void __launch_bounds__(kTopMax) ppr_topk_sort_kernel(int kk, int top, int c0, int* __restrict__ ids,
                                                                float* __restrict__ vals) {
    __shared__ unsigned s_key[kTopMax];
    __shared__ int s_id[kTopMax];
    const size_t row = static_cast<size_t>(c0 + blockIdx.x) * top;
    const int i = threadIdx.x;
    int id = -1;
    float v = 0.0f;
    if (i < kk) {
        id = ids[row + i];
        v = vals[row + i];
        s_key[i] = dev::order_key(v);
        s_id[i] = id;
    }
    __syncthreads();  // every entry is read before any is moved
    if (i < kk) {
        const unsigned key = s_key[i];
        int place = 0;
        for (int j = 0; j < kk; ++j) place += s_key[j] > key || (s_key[j] == key && s_id[j] < id);
        ids[row + place] = id;
        vals[row + place] = v;
    } else if (i < top) {
        ids[row + i] = -1;
        vals[row + i] = 0.0f;
    }
}

int run_top_k(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, int k, const int* offsets,
              const int* nodes, const float* weights, int top, int* d_ids, float* d_vals, int* iterations,
              float* final_residual, bool* converged, float* l2_history, int history_capacity) {
    if (top < 1 || top > kTopMax || !d_ids || !d_vals) return SPMV_B200_INVALID_ARGUMENT;
    const long long n = adj ? adj->num_rows : 0;
    const int kk = static_cast<int>(std::min<long long>(top, n));
    const int tie_blocks = static_cast<int>((n + kTieChunk - 1) / kTieChunk);
    Device sel, hist, ties;  // allocated with the first chunk, once the inputs are validated
    return run_chunks(
        adj, config, k, offsets, nodes, weights, iterations, final_residual, converged, l2_history, history_capacity,
        [&](const float* fin, const double* block_sums, int blocks, int c0, int width, cudaStream_t stream) {
            if (!sel.p && !(sel.alloc(sizeof(Select)) && hist.alloc(sizeof(unsigned) * kW * 256) &&
                            ties.alloc(sizeof(int) * kW * static_cast<size_t>(tie_blocks)))) {
                cudaGetLastError();
                return static_cast<int>(SPMV_B200_CUDA_MALLOC);
            }
            Select* s = sel.as<Select>();
            ppr_topk_begin_kernel<<<1, kSel, 0, stream>>>(block_sums, blocks, s, hist.as<unsigned>());
            const int hist_grid = grid_for(n, kSel, kSelBlocksMax);
            for (int shift = 24; shift >= 0; shift -= 8) {
                ppr_topk_hist_kernel<<<hist_grid, kSel, 0, stream>>>(fin, n, width, shift, s, hist.as<unsigned>());
                ppr_topk_bin_kernel<<<1, kW * 32, 0, stream>>>(hist.as<unsigned>(), shift, kk, width, s);
            }
            ppr_topk_above_kernel<<<tie_blocks, kSel, 0, stream>>>(fin, n, width, s, top, c0, d_ids, d_vals,
                                                                   ties.as<int>());
            ppr_topk_tie_scan_kernel<<<width, kSel, 0, stream>>>(ties.as<int>(), tie_blocks);
            ppr_topk_tie_write_kernel<<<tie_blocks, kSel, 0, stream>>>(fin, n, width, s, ties.as<int>(), kk, top, c0,
                                                                       d_ids, d_vals);
            ppr_topk_sort_kernel<<<width, kTopMax, 0, stream>>>(kk, top, c0, d_ids, d_vals);
            counted(13);
            return 0;
        });
}

}  // namespace ppr
}  // namespace b200
}  // namespace spmv

extern "C" {

int spmv_b200_pagerank_personalized_batch_top_k(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                                int k, const int* offsets, const int* nodes, const float* weights,
                                                int top, int* d_ids, float* d_vals, int* iterations,
                                                float* final_residual, bool* converged, float* l2_history,
                                                int history_capacity) {
    try {
        return spmv::b200::ppr::run_top_k(adj, config, k, offsets, nodes, weights, top, d_ids, d_vals, iterations,
                                          final_residual, converged, l2_history, history_capacity);
    } catch (...) {
        return SPMV_B200_OUT_OF_MEMORY;
    }
}

unsigned long long spmv_b200_ppr_topk_launch_count(void) { return spmv::b200::ppr::g_launches.load(); }

}  // extern "C"
