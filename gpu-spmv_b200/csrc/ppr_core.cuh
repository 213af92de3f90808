// ppr_core.cuh -- the chunk loop of batched personalized PageRank, shared by libspmv_b200_ppr.so
// (ppr_batch.cu: dense [n][k] ranks) and libspmv_b200_ppr_topk.so (ppr_topk.cu: each column's top K).
//
// k personalized PageRank vectors of one graph advance together, in chunks of kW = 8 columns.
// A chunk's vectors are stored node-major, r[node][0..8), 32 bytes per node: the PageRank product is
// bound by the L2's random-sector rate (DESIGN.md section 8), and one gather of r_old[col] is then one
// aligned sector that carries all 8 values.  One iteration of a chunk:
//   ppr_step_kernel    nnz-balanced merge-path tiles (persistent CTAs, static tile assignment): the
//                      tile's (column, value) stream is read once, each non-zero gathers 32 bytes and
//                      multiplies all 8 lanes, rows are summed per lane in a fixed order, and the
//                      personalized update (dev::pr_row_value) is applied per lane with f64 sums of
//                      delta^2, |delta| and the next dangling mass.  A frozen lane copies r_old.
//   ppr_fixup_kernel   rows open at a tile end: the carries of the run of tiles, in tile order (no atomics).
//   ppr_reduce_kernel  one CTA folds the per-CTA sums per lane and makes each lane's stop decision:
//                      iteration count, residual, history entry, next dangling mass; a lane that met the
//                      tolerance is frozen from the next iteration on.  The number of active lanes is the
//                      only thing the host reads, one iteration late.
// The decomposition (tiles, persistent grid, fix-up grid) depends only on the matrix and the device, never on
// k or on a column's lane, and every lane runs the same operations: a column's result is bit-identical
// wherever it sits in the batch.  After the loop, ppr_sum_kernel takes per-CTA f64 sums of every lane and the
// caller's finishing step turns the chunk into its output; both outputs normalise a value with
// normalised(v, lane_total(...)), so they agree bit for bit.
//
// The dangling set comes from libspmv_b200.so's public building blocks (pr_plan_create -> pr_colsum ->
// pr_dangling_bits), so the rule for which node is dangling lives in one place.
//
// Each library compiles this header in exactly one translation unit; g_launches is that library's counter.
#pragma once
#include "merge_rows.cuh"
#include "spmv_b200.h"

#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <vector>

namespace spmv {
namespace b200 {
namespace ppr {

constexpr int kW = 8;                 // columns per chunk (32 bytes per node)
constexpr int kBT = 256;              // threads of the step kernel
constexpr int kBIPT = 5;              // merge items per thread (odd: see kMergeItemsPerThread)
constexpr int kBTile = kBT * kBIPT;   // merge items per tile
constexpr int kSums = 3 * kW;         // per lane: sum delta^2, sum |delta|, dangling mass
constexpr int kFixBlocksMax = 148 * 8;
constexpr int kNormBlocksMax = 148 * 8;

std::atomic<unsigned long long> g_launches{0};
inline void counted(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }

// Per-chunk loop state, device-resident; written by ppr_state_init_kernel and ppr_reduce_kernel only.
struct State {
    float dsum[kW];       // dangling mass of r_old per lane
    float residual[kW];   // L2 norm of the delta of the lane's last active iteration
    int iters[kW];        // iterations the lane ran
    unsigned frozen;      // bit c: lane c copies r_old through (converged, or not a column of the batch)
    unsigned converged;
    int active;           // lanes still iterating
    int iter;             // iterations completed by the chunk
};

__device__ __forceinline__ void load8(const float* p, float (&v)[kW]) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    const float4 b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(float* p, const float (&v)[kW]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
// the gather of r_old[col]: one aligned 32-byte sector, read-only path
__device__ __forceinline__ void gather8(const float* p, float (&v)[kW]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + 4));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

struct StepArgs {
    const float* r_old;   // [n][kW]
    float* r_new;         // [n][kW]
    const float* vhat;    // [n][kW] normalised personalization vectors
    const uint32_t* bits; // dangling bitmask
    const State* st;
    float damping;
    float teleport;       // 1 - d, as pr_step sets it for the personalized form
    int n;
};

// The personalized update of one row for every lane, from its 8 raw row sums (in y, replaced by the
// new ranks), and the row's contribution to the lane sums.
__device__ __forceinline__ void update_row(const StepArgs& a, int row, float (&y)[kW], const float (&ctx)[kW],
                                           unsigned frozen, double (&s)[kSums]) {
    const size_t base = static_cast<size_t>(row) * kW;
    float old[kW];
    gather8(a.r_old + base, old);
    const bool dangling = (__ldg(a.bits + (row >> 5)) >> (row & 31)) & 1u;
#pragma unroll
    for (int c = 0; c < kW; ++c) {
        const float v = ((frozen >> c) & 1u) ? old[c] : dev::pr_row_value(a.damping, y[c], ctx[c], a.teleport, a.vhat + base + c, 0);
        y[c] = v;
        const double diff = static_cast<double>(v) - static_cast<double>(old[c]);
        s[c] += diff * diff;
        s[kW + c] += fabs(diff);
        if (dangling) s[2 * kW + c] += static_cast<double>(v);
    }
    store8(a.r_new + base, y);
}

// block-wide sum of the kSums lane sums into out[0 .. kSums) (fixed order)
template <int THREADS>
__device__ __forceinline__ void block_store_sums(double (&s)[kSums], double* __restrict__ out, double (*scratch)[kSums]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < kSums; ++j) {
        const double t = dev::warp_sum(s[j]);
        if (lane == 0) scratch[warp][j] = t;
    }
    __syncthreads();
    if (threadIdx.x < kSums) {
        double t = 0.0;
        for (int w = 0; w < THREADS / 32; ++w) t += scratch[w][threadIdx.x];
        out[threadIdx.x] = t;
    }
}

__global__ void ppr_partition_kernel(int rows, int nnz, const int* __restrict__ row_ptrs, int num_tiles,
                                     int2* __restrict__ coords) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > num_tiles) return;
    const long long total = static_cast<long long>(rows) + nnz;
    const long long d = static_cast<long long>(t) * kBTile;
    coords[t] = diagonal_search_global(static_cast<int>(d < total ? d : total), row_ptrs, rows, nnz);
}

// ------------------------------------------------------------------------------------------ step ----
__global__ void __launch_bounds__(kBT)
ppr_step_kernel(int rows, int nnz, const int* __restrict__ row_ptrs, const int* __restrict__ col_indices,
                const float* __restrict__ values, const int2* __restrict__ coords, int num_tiles, StepArgs a,
                int* __restrict__ carry_row, float* __restrict__ carry_val, double* __restrict__ partials) {
    __shared__ __align__(16) float s_prod[kBTile * kW];  // the tile's products, 8 lanes per non-zero
    __shared__ int s_end[kBTile + 1];                    // global END offset of tile-local row i
    __shared__ float s_warp_val[kBT / 32][kW];
    __shared__ int s_warp_flag[kBT / 32];
    __shared__ double s_sums[kBT / 32][kSums];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned frozen = a.st->frozen;
    float ctx[kW];
#pragma unroll
    for (int c = 0; c < kW; ++c) ctx[c] = dev::pr_step_context(a.damping, a.st->dsum[c], a.n, a.vhat);
    double sums[kSums];
#pragma unroll
    for (int j = 0; j < kSums; ++j) sums[j] = 0.0;

    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int2 c0 = coords[tile];
        const int2 c1 = coords[tile + 1];
        const int row_s = c0.x, nz_s = c0.y, nz_e = c1.y;
        const int tile_rows = c1.x - c0.x;
        const int tile_nz = c1.y - c0.y;
        const int tile_items = tile_rows + tile_nz;

        for (int i = tid; i <= tile_rows; i += kBT)
            s_end[i] = (row_s + i < rows) ? dev::ld_stream_i(row_ptrs + row_s + 1 + i) : INT_MAX;
        // the matrix stream of the tile, read once for all lanes: one 32-byte gather per non-zero
#pragma unroll 2
        for (int j = nz_s + tid; j < nz_e; j += kBT) {
            const float w = dev::ld_stream_f(values + j);
            float x[kW];
            gather8(a.r_old + static_cast<size_t>(dev::ld_stream_i(col_indices + j)) * kW, x);
#pragma unroll
            for (int c = 0; c < kW; ++c) x[c] = w * x[c];
            store8(s_prod + (j - nz_s) * kW, x);
        }
        const bool first_row_split = (row_s < rows) && (nz_s > __ldg(row_ptrs + row_s));
        __syncthreads();

        // per-thread diagonal inside the tile
        const int diag = min(tid * kBIPT, tile_items);
        int lo = max(diag - tile_nz, 0);
        int hi = min(diag, tile_rows);
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (s_end[mid] <= nz_s + (diag - mid - 1)) lo = mid + 1;
            else hi = mid;
        }
        int r = lo;
        int z = nz_s + (diag - lo);
        const int my_items = min(kBIPT, tile_items - diag);

        float running[kW], first_sum[kW];
#pragma unroll
        for (int c = 0; c < kW; ++c) running[c] = first_sum[c] = 0.0f;
        bool emitted = false;
        int first_row = 0;
        int row_end = s_end[r];
#pragma unroll
        for (int it = 0; it < kBIPT; ++it) {
            if (it < my_items) {
                if (z < row_end) {
                    float p[kW];
                    load8(s_prod + (z - nz_s) * kW, p);
#pragma unroll
                    for (int c = 0; c < kW; ++c) running[c] += p[c];
                    ++z;
                } else {
                    if (!emitted) {  // may still need the carry of earlier threads
                        emitted = true;
                        first_row = r;
#pragma unroll
                        for (int c = 0; c < kW; ++c) first_sum[c] = running[c];
                    } else {         // raw row sum; the update is applied after the tile (below)
                        store8(a.r_new + static_cast<size_t>(row_s + r) * kW, running);
                    }
#pragma unroll
                    for (int c = 0; c < kW; ++c) running[c] = 0.0f;
                    ++r;
                    row_end = s_end[r];
                }
            }
        }

        // segmented scan of (emitted, running) over the CTA, lane by lane
        float v[kW], ex_v[kW];
        int f = 0, ex_f = 0;
#pragma unroll
        for (int c = 0; c < kW; ++c) {
            v[c] = running[c];
            warp_segmented_scan(v[c], emitted, lane, f, ex_v[c], ex_f);
        }
        if (lane == 31) {
#pragma unroll
            for (int c = 0; c < kW; ++c) s_warp_val[warp][c] = v[c];
            s_warp_flag[warp] = f;
        }
        __syncthreads();
        float pre_v[kW];
#pragma unroll
        for (int c = 0; c < kW; ++c) pre_v[c] = 0.0f;
        for (int w = 0; w < warp; ++w) {
            const int wf = s_warp_flag[w];
#pragma unroll
            for (int c = 0; c < kW; ++c) pre_v[c] = wf ? s_warp_val[w][c] : pre_v[c] + s_warp_val[w][c];
        }
        if (emitted) {
            float total[kW];
#pragma unroll
            for (int c = 0; c < kW; ++c) total[c] = (ex_f ? ex_v[c] : pre_v[c] + ex_v[c]) + first_sum[c];
            // the first row of a split row is parked raw for the fix-up; every other row is stored raw too
            store8(a.r_new + static_cast<size_t>(row_s + first_row) * kW, total);
        }
        if (tid == kBT - 1) {  // the row still open at the tile end
            const int row_e = c1.x;
            const int open_start = tile_rows > 0 ? s_end[tile_rows - 1] : (row_s < rows ? __ldg(row_ptrs + row_s) : nz_e);
            const bool has_open = (row_e < rows) && (nz_e > max(open_start, nz_s));
            carry_row[tile] = has_open ? row_e : -1;
#pragma unroll
            for (int c = 0; c < kW; ++c) carry_val[static_cast<size_t>(tile) * kW + c] = has_open ? (f ? v[c] : pre_v[c] + v[c]) : 0.0f;
        }
        __syncthreads();  // every raw row sum of the tile is visible CTA-wide

        // update of the rows this tile finished (a split first row is the fix-up's)
        const int g0 = row_s + (first_row_split ? 1 : 0), g1 = c1.x;
        for (int g = g0 + tid; g < g1; g += kBT) {
            float y[kW];
            load8(a.r_new + static_cast<size_t>(g) * kW, y);
            update_row(a, g, y, ctx, frozen, sums);
        }
        __syncthreads();  // s_prod / s_end are reused by the next tile
    }
    block_store_sums<kBT>(sums, partials + static_cast<size_t>(blockIdx.x) * kSums, s_sums);
}

// ----------------------------------------------------------------------------------------- fix-up ----
__global__ void __launch_bounds__(256)
ppr_fixup_kernel(int num_tiles, const int* __restrict__ carry_row, const float* __restrict__ carry_val, StepArgs a,
                 double* __restrict__ partials) {
    __shared__ double s_sums[256 / 32][kSums];
    const unsigned frozen = a.st->frozen;
    float ctx[kW];
#pragma unroll
    for (int c = 0; c < kW; ++c) ctx[c] = dev::pr_step_context(a.damping, a.st->dsum[c], a.n, a.vhat);
    double sums[kSums];
#pragma unroll
    for (int j = 0; j < kSums; ++j) sums[j] = 0.0;
    for (int t = blockIdx.x * 256 + threadIdx.x; t < num_tiles; t += gridDim.x * 256) {
        const int row = carry_row[t];
        if (row < 0 || (t > 0 && carry_row[t - 1] == row)) continue;  // not the leader of a run of tiles
        float total[kW];
#pragma unroll
        for (int c = 0; c < kW; ++c) total[c] = carry_val[static_cast<size_t>(t) * kW + c];
        for (int u = t + 1; u < num_tiles && carry_row[u] == row; ++u)
#pragma unroll
            for (int c = 0; c < kW; ++c) total[c] += carry_val[static_cast<size_t>(u) * kW + c];
        // the tile in which the row ends parked its own share
        float y[kW];
        load8(a.r_new + static_cast<size_t>(row) * kW, y);
#pragma unroll
        for (int c = 0; c < kW; ++c) y[c] = y[c] + total[c];
        update_row(a, row, y, ctx, frozen, sums);
    }
    block_store_sums<256>(sums, partials + static_cast<size_t>(blockIdx.x) * kSums, s_sums);
}

// ----------------------------------------------------------------------------- reduce and stop rule ----
// One CTA: the lane sums of all `count` partial rows, in a fixed order, then each lane's stop decision.
__global__ void __launch_bounds__(256)
ppr_reduce_kernel(const double* __restrict__ partials, int count, State* __restrict__ st, float tolerance,
                  float* __restrict__ history, int capacity) {
    __shared__ double s_sums[256 / 32][kSums];
    __shared__ double s_tot[kSums];
    double s[kSums];
#pragma unroll
    for (int j = 0; j < kSums; ++j) s[j] = 0.0;
    for (int i = threadIdx.x; i < count; i += 256)
#pragma unroll
        for (int j = 0; j < kSums; ++j) s[j] += partials[static_cast<size_t>(i) * kSums + j];
    block_store_sums<256>(s, s_tot, s_sums);
    __syncthreads();
    const int c = threadIdx.x;
    const int it = st->iter + 1;  // the iteration these sums belong to
    const unsigned frozen = st->frozen;
    bool newly = false;
    if (c < kW && !((frozen >> c) & 1u)) {
        const float residual = sqrtf(static_cast<float>(s_tot[c]));  // L2 norm of the delta
        st->residual[c] = residual;
        st->iters[c] = it;
        st->dsum[c] = static_cast<float>(s_tot[2 * kW + c]);
        if (history && it <= capacity) history[static_cast<size_t>(c) * capacity + it - 1] = residual;
        newly = residual < tolerance;
    }
    const unsigned now = __ballot_sync(0xffffffffu, newly);
    __syncthreads();  // every lane has read st->iter and st->frozen
    if (threadIdx.x == 0) {
        st->frozen = frozen | now;
        st->converged |= now;
        st->active = kW - __popc((frozen | now) & ((1u << kW) - 1u));
        st->iter = it;
    }
}

// ----------------------------------------------------------------------------------------- set-up ----
__global__ void ppr_init_ranks_kernel(long long n, float init, float* __restrict__ r) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float4 v = make_float4(init, init, init, init);
        *reinterpret_cast<float4*>(r + i * kW) = v;
        *reinterpret_cast<float4*>(r + i * kW + 4) = v;
    }
}

// vhat[node][lane] = value for the m listed entries of the chunk (the rest is zero)
__global__ void ppr_scatter_kernel(int m, const int* __restrict__ node, const int* __restrict__ lane,
                                   const float* __restrict__ value, float* __restrict__ vhat) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x)
        vhat[static_cast<size_t>(node[j]) * kW + lane[j]] = value[j];
}

// D_0 = (float)(#dangling * (1/n)) for every lane, as pr_init computes it; lanes outside `live` are frozen
__global__ void __launch_bounds__(1024) ppr_state_init_kernel(const uint32_t* __restrict__ bits, int n, unsigned live,
                                                              State* __restrict__ st) {
    __shared__ unsigned s[32];
    const int words = (n + 31) / 32;
    unsigned cnt = 0;
    for (int w = threadIdx.x; w < words; w += 1024) {
        const int lim = min(32, n - w * 32);
        const uint32_t mask = lim == 32 ? 0xffffffffu : ((1u << lim) - 1u);
        cnt += __popc(bits[w] & mask);
    }
    cnt = dev::warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x < kW) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += static_cast<double>(s[w]);
        const float init = 1.0f / n;
        st->dsum[threadIdx.x] = static_cast<float>(t * static_cast<double>(init));
        st->residual[threadIdx.x] = 0.0f;
        st->iters[threadIdx.x] = 0;
    }
    if (threadIdx.x == 0) {
        st->frozen = ~live & ((1u << kW) - 1u);
        st->converged = 0;
        st->active = __popc(live);
        st->iter = 0;
    }
}

// ------------------------------------------------------------------------------------- normalise ----
// per-CTA f64 sums of every lane of r
__global__ void __launch_bounds__(256) ppr_sum_kernel(const float* __restrict__ r, long long n, double* __restrict__ block_sums) {
    __shared__ double s[256 / 32][kW];
    double acc[kW];
#pragma unroll
    for (int c = 0; c < kW; ++c) acc[c] = 0.0;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256) {
        float v[kW];
        load8(r + i * kW, v);
#pragma unroll
        for (int c = 0; c < kW; ++c) acc[c] += static_cast<double>(v[c]);
    }
#pragma unroll
    for (int c = 0; c < kW; ++c) {
        const double t = dev::warp_sum(acc[c]);
        if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5][c] = t;
    }
    __syncthreads();
    if (threadIdx.x < kW) {
        double t = 0.0;
        for (int w = 0; w < 256 / 32; ++w) t += s[w][threadIdx.x];
        block_sums[static_cast<size_t>(blockIdx.x) * kW + threadIdx.x] = t;
    }
}

// The f32 total of lane c from ppr_sum_kernel's per-CTA sums (f64, CTA order) and a value normalised by it,
// as spmv_b200_pr_normalize does.
__device__ __forceinline__ float lane_total(const double* __restrict__ block_sums, int blocks, int c) {
    double t = 0.0;
    for (int b = 0; b < blocks; ++b) t += block_sums[static_cast<size_t>(b) * kW + c];
    return static_cast<float>(t);
}
__device__ __forceinline__ float normalised(float v, float t) { return t > 0.0f ? __fdiv_rn(v, t) : v; }

// ------------------------------------------------------------------------------------------- host ----
inline int grid_for(long long items, int per_block, int cap) {
    long long b = (items + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return static_cast<int>(b < cap ? b : cap);
}

// Host-side validation and normalisation of one column: v = w / sum(w), f64 sum in index order.
inline int normalise_column(int n, const int* nodes, const float* weights, int lo, int hi, std::vector<float>* out) {
    double sum = 0.0;
    for (int j = lo; j < hi; ++j) {
        if (nodes[j] < 0 || nodes[j] >= n || (j > lo && nodes[j] <= nodes[j - 1])) return SPMV_B200_INVALID_ARGUMENT;
        const float w = weights ? weights[j] : 1.0f;
        if (!std::isfinite(w) || w < 0.0f) return SPMV_B200_INVALID_ARGUMENT;
        sum += static_cast<double>(w);
    }
    if (sum == 0.0) return SPMV_B200_INVALID_ARGUMENT;
    out->resize(static_cast<size_t>(hi - lo));
    for (int j = lo; j < hi; ++j) (*out)[j - lo] = static_cast<float>(static_cast<double>(weights ? weights[j] : 1.0f) / sum);
    return 0;
}

struct Device {
    void* p = nullptr;
    ~Device() { cudaFree(p); }
    template <class T> T* as() const { return static_cast<T*>(p); }
    bool alloc(size_t bytes) { return cudaMalloc(&p, bytes > 0 ? bytes : 1) == cudaSuccess; }
};

// The chunk loop: validation, dangling set, partition, then per chunk of kW columns the scatter and init, the
// iterations and the per-lane sums of the final vector, after which `finish` turns the chunk into the caller's
// output.  finish(fin, block_sums, blocks, c0, width, stream) enqueues its kernels on `stream` after the sums
// (fin: the chunk's [n][kW] final vector; block_sums: [blocks][kW] f64 per-CTA sums, see lane_total; lanes
// [0, width) are columns c0 .. c0 + width) and returns 0 or a status; it must not wait on the host.
template <class Finish>
int run_chunks(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, int k, const int* offsets,
               const int* nodes, const float* weights, int* iterations, float* final_residual, bool* converged,
               float* l2_history, int history_capacity, Finish&& finish) {
    if (!adj || !offsets || !iterations || !final_residual || !converged || k <= 0 || history_capacity < 0 ||
        (history_capacity > 0 && !l2_history))
        return SPMV_B200_INVALID_ARGUMENT;
    const spmv_b200_pagerank_config defaults{0.85f, 1e-6f, 100};
    if (!config) config = &defaults;
    const int n = adj->num_rows;
    if (offsets[0] != 0) return SPMV_B200_INVALID_ARGUMENT;
    for (int c = 0; c < k; ++c)
        if (offsets[c + 1] < offsets[c]) return SPMV_B200_INVALID_ARGUMENT;
    if (offsets[k] > 0 && !nodes) return SPMV_B200_INVALID_ARGUMENT;
    std::vector<std::vector<float>> vhat(static_cast<size_t>(k));
    for (int c = 0; c < k; ++c) {
        const int rc = normalise_column(n, nodes, weights, offsets[c], offsets[c + 1], &vhat[c]);
        if (rc != 0) return rc;
    }
    for (int c = 0; c < k; ++c) {
        iterations[c] = 0;
        final_residual[c] = 0.0f;
        converged[c] = false;
    }
    // non-square adjacency: the single-vector path's INVALID_DIMENSION (reference src/pagerank.cu:102-107)
    if (adj->num_cols != n) return SPMV_B200_INVALID_DIMENSION;

    cudaStream_t stream = nullptr;
    // the dangling set, from libspmv_b200.so's building blocks
    spmv_b200_pr_plan* plan = nullptr;
    int rc = spmv_b200_pr_plan_create(adj, 0, n, stream, &plan);
    if (rc != 0) return rc;
    struct PlanGuard {
        spmv_b200_pr_plan* p;
        ~PlanGuard() { spmv_b200_pr_plan_destroy(p); }
    } plan_guard{plan};
    const int nnz = adj->nnz;
    const int num_tiles = static_cast<int>((static_cast<long long>(n) + nnz + kBTile - 1) / kBTile);
    int dev_id = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppr_step_kernel, kBT, 0);
    const int step_grid = std::max(1, std::min(num_tiles, std::max(1, sms * std::max(per_sm, 1))));
    const int fix_grid = grid_for(num_tiles, 256, kFixBlocksMax);
    const int norm_grid = grid_for(n, 256, kNormBlocksMax);
    const size_t vec_bytes = sizeof(float) * kW * static_cast<size_t>(n);
    const size_t words = (static_cast<size_t>(n) + 31) / 32;
    size_t max_entries = 0;
    for (int c0 = 0; c0 < k; c0 += kW)
        max_entries = std::max(max_entries, static_cast<size_t>(offsets[std::min(k, c0 + kW)] - offsets[c0]));
    Device colsum, bits, coords, carry_row, carry_val, partials, ra, rb, vh, state, hist, ent_node, ent_lane, ent_val, norm;
    const bool ok = colsum.alloc(sizeof(double) * n) && bits.alloc(sizeof(uint32_t) * words) &&
                    coords.alloc(sizeof(int2) * (static_cast<size_t>(num_tiles) + 1)) &&
                    carry_row.alloc(sizeof(int) * num_tiles) && carry_val.alloc(sizeof(float) * kW * num_tiles) &&
                    partials.alloc(sizeof(double) * kSums * (step_grid + fix_grid)) && ra.alloc(vec_bytes) &&
                    rb.alloc(vec_bytes) && vh.alloc(vec_bytes) && state.alloc(sizeof(State)) &&
                    hist.alloc(sizeof(float) * kW * static_cast<size_t>(history_capacity)) &&
                    ent_node.alloc(sizeof(int) * max_entries) && ent_lane.alloc(sizeof(int) * max_entries) &&
                    ent_val.alloc(sizeof(float) * max_entries) && norm.alloc(sizeof(double) * kW * norm_grid);
    if (!ok) {
        cudaGetLastError();
        return SPMV_B200_CUDA_MALLOC;
    }
    auto launch_failed = [] { return cudaGetLastError() != cudaSuccess; };
    // dangling nodes: columns whose stored values sum to 0
    cudaMemsetAsync(colsum.p, 0, sizeof(double) * n, stream);
    if ((rc = spmv_b200_pr_colsum(plan, colsum.as<double>(), stream)) != 0) return rc;
    if ((rc = spmv_b200_pr_dangling_bits(colsum.as<double>(), n, bits.as<uint32_t>(), stream)) != 0) return rc;
    ppr_partition_kernel<<<(num_tiles + 1 + 255) / 256, 256, 0, stream>>>(n, nnz, adj->d_row_ptrs, num_tiles,
                                                                          coords.as<int2>());
    counted(1);
    if (launch_failed()) return SPMV_B200_KERNEL_LAUNCH;

    int* h_active = nullptr;
    if (cudaMallocHost(&h_active, 2 * sizeof(int)) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_CUDA_MALLOC;
    }
    struct HostGuard {
        int* p;
        ~HostGuard() { cudaFreeHost(p); }
    } host_guard{h_active};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
    struct EventGuard {
        cudaEvent_t* e;
        ~EventGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); }
    } event_guard{ev};

    std::vector<int> h_node, h_lane;
    std::vector<float> h_val, h_hist;
    State h_state;
    for (int c0 = 0; c0 < k && rc == 0; c0 += kW) {
        const int width = std::min(kW, k - c0);
        // the chunk's normalised vectors, node-major
        h_node.clear(); h_lane.clear(); h_val.clear();
        for (int c = 0; c < width; ++c)
            for (int j = offsets[c0 + c]; j < offsets[c0 + c + 1]; ++j) {
                h_node.push_back(nodes[j]);
                h_lane.push_back(c);
                h_val.push_back(vhat[c0 + c][j - offsets[c0 + c]]);
            }
        const int m = static_cast<int>(h_node.size());
        cudaMemsetAsync(vh.p, 0, vec_bytes, stream);
        if (cudaMemcpyAsync(ent_node.p, h_node.data(), sizeof(int) * m, cudaMemcpyHostToDevice, stream) != cudaSuccess ||
            cudaMemcpyAsync(ent_lane.p, h_lane.data(), sizeof(int) * m, cudaMemcpyHostToDevice, stream) != cudaSuccess ||
            cudaMemcpyAsync(ent_val.p, h_val.data(), sizeof(float) * m, cudaMemcpyHostToDevice, stream) != cudaSuccess) {
            cudaGetLastError();
            return SPMV_B200_CUDA_MEMCPY;
        }
        ppr_scatter_kernel<<<grid_for(m, 256, kNormBlocksMax), 256, 0, stream>>>(m, ent_node.as<int>(), ent_lane.as<int>(),
                                                                                ent_val.as<float>(), vh.as<float>());
        ppr_init_ranks_kernel<<<grid_for(n, 256, kNormBlocksMax), 256, 0, stream>>>(n, 1.0f / n, ra.as<float>());
        ppr_state_init_kernel<<<1, 1024, 0, stream>>>(bits.as<uint32_t>(), n, (1u << width) - 1u, state.as<State>());
        counted(3);
        if (launch_failed()) return SPMV_B200_KERNEL_LAUNCH;
        // host pointers are dropped at the end of the iteration; the copies above must have read them
        if (cudaStreamSynchronize(stream) != cudaSuccess) {
            cudaGetLastError();
            return SPMV_B200_CUDA_MEMCPY;
        }

        StepArgs a;
        a.vhat = vh.as<float>();
        a.bits = bits.as<uint32_t>();
        a.st = state.as<State>();
        a.damping = config->damping_factor;
        a.teleport = 1.0f - config->damping_factor;
        a.n = n;
        float* r_old = ra.as<float>();
        float* r_new = rb.as<float>();
        const float* fin = r_old;  // the initial vector when the loop never runs
        int pending = -1;          // slot of the iteration whose active count is still in flight
        for (int it = 0; it < config->max_iterations; ++it) {
            const int slot = it & 1;
            a.r_old = r_old;
            a.r_new = r_new;
            ppr_step_kernel<<<step_grid, kBT, 0, stream>>>(n, nnz, adj->d_row_ptrs, adj->d_col_indices, adj->d_values,
                                                           coords.as<int2>(), num_tiles, a, carry_row.as<int>(),
                                                           carry_val.as<float>(), partials.as<double>());
            ppr_fixup_kernel<<<fix_grid, 256, 0, stream>>>(num_tiles, carry_row.as<int>(), carry_val.as<float>(), a,
                                                           partials.as<double>() + static_cast<size_t>(step_grid) * kSums);
            ppr_reduce_kernel<<<1, 256, 0, stream>>>(partials.as<double>(), step_grid + fix_grid, state.as<State>(),
                                                     config->tolerance, history_capacity > 0 ? hist.as<float>() : nullptr,
                                                     history_capacity);
            counted(3);
            if (launch_failed()) {
                rc = SPMV_B200_KERNEL_LAUNCH;
                break;
            }
            cudaMemcpyAsync(h_active + slot, &state.as<State>()->active, sizeof(int), cudaMemcpyDeviceToHost, stream);
            cudaEventRecord(ev[slot], stream);
            fin = r_new;  // frozen lanes are carried through: the last vector written holds every lane's result
            std::swap(r_old, r_new);
            // the stop rule, one iteration late: iteration it - 1's count is read while iteration it is queued
            if (pending >= 0) {
                if (cudaEventSynchronize(ev[pending]) != cudaSuccess) {
                    cudaGetLastError();
                    rc = SPMV_B200_KERNEL_LAUNCH;
                    break;
                }
                if (h_active[pending] == 0) break;
            }
            pending = slot;
        }
        if (rc != 0) break;
        ppr_sum_kernel<<<norm_grid, 256, 0, stream>>>(fin, n, norm.as<double>());
        counted(1);
        if (launch_failed()) return SPMV_B200_KERNEL_LAUNCH;
        if ((rc = finish(fin, norm.as<double>(), norm_grid, c0, width, stream)) != 0) return rc;
        if (launch_failed()) return SPMV_B200_KERNEL_LAUNCH;
        if (cudaMemcpyAsync(&h_state, state.p, sizeof(State), cudaMemcpyDeviceToHost, stream) != cudaSuccess) {
            cudaGetLastError();
            return SPMV_B200_CUDA_MEMCPY;
        }
        if (history_capacity > 0) {
            h_hist.resize(static_cast<size_t>(kW) * history_capacity);
            cudaMemcpyAsync(h_hist.data(), hist.p, sizeof(float) * h_hist.size(), cudaMemcpyDeviceToHost, stream);
        }
        if (cudaStreamSynchronize(stream) != cudaSuccess) {
            cudaGetLastError();
            return SPMV_B200_KERNEL_LAUNCH;
        }
        for (int c = 0; c < width; ++c) {
            iterations[c0 + c] = h_state.iters[c];
            final_residual[c0 + c] = h_state.residual[c];
            converged[c0 + c] = (h_state.converged >> c) & 1u;
            for (int i = 0; i < std::min(h_state.iters[c], history_capacity); ++i)
                l2_history[static_cast<size_t>(c0 + c) * history_capacity + i] = h_hist[static_cast<size_t>(c) * history_capacity + i];
        }
    }
    cudaStreamSynchronize(stream);
    return rc;
}

}  // namespace ppr
}  // namespace b200
}  // namespace spmv
