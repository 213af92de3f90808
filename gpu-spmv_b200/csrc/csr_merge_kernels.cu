// csr_merge_kernels.cu -- two-level merge-path CSR SpMV for sm_100a, and the
// fused PageRank iteration built on it.
//
// Replaces merge_path_search + spmv_csr_merge_path_kernel + the pre-launch
// cudaMemset (reference src/spmv_kernels.cu:48-72, :75-130, :267).  The
// reference gives every THREAD its own diagonal (two global binary searches
// per thread), walks its non-zeros uncoalesced and commits rows with float
// atomics; its search is also off by one (SURVEY F3), so its results are
// wrong.  This implementation uses the canonical Merrill-Garland formulation:
//
//   level 1  merge_partition_kernel: one search per TILE of kMergeTile merge
//            items (rows + nnz are the two merged lists) -> coords[].
//   level 2  merge_tile_kernel: a CTA takes one tile.  It stages the tile's
//            row-end offsets in shared memory, streams the tile's contiguous
//            non-zero range with coalesced 128-bit loads of values and
//            col_indices, gathers x and parks the products in shared memory.
//            Every thread then locates its own diagonal by a binary search IN
//            SHARED MEMORY and consumes kMergeItemsPerThread items serially.
//            Rows that start inside a thread are finished by that thread; the
//            row open at a thread boundary is resolved by a warp-shuffle
//            segmented scan over (emitted?, carry) pairs plus an 8-entry
//            cross-warp fold.  The row left open at the tile end goes to
//            carry_row/carry_val.
//   level 3  merge_fixup_kernel: for every run of tiles that left the same row
//            open, one thread adds the run's carries (in tile order) to that
//            row.  No float atomics and no pre-zeroing of y: every row is
//            written exactly once by level 2 and touched by at most one
//            thread of level 3, so results are deterministic.
//
// The row epilogue is a template parameter.  PlainRow writes y.  PageRankRow
// applies r_new = (d*y + d*dangling/n) + (1-d)/n in the reference's operation
// order (src/pagerank.cu:111-114), and accumulates sum (r_new-r_old)^2,
// sum |r_new-r_old| and the next iteration's dangling mass in f64 -- SpMV,
// damping/teleport, dangling mass and residual in ONE pass over the matrix.
//
// Roofline: HBM.  Algorithmic bytes per launch = 8*nnz + 4*(rows+1) + 4*cols +
// 4*rows (reference src/bandwidth.cpp:34-42); merge-path timing includes
// partition + tile + fix-up, as the reference's includes its memset.
#include "merge_rows.cuh"

#include <climits>

namespace spmv {
namespace b200 {

// ------------------------------------------------------------ plan layout ----

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int fixup_blocks_for(int num_tiles) { return (num_tiles + 255) / 256; }

size_t merge_plan_bytes(int rows, int nnz, bool with_partials) {
    const size_t tiles = static_cast<size_t>(merge_num_tiles(rows, nnz));
    size_t b = align_up((tiles + 1) * sizeof(int2), 256);
    b += align_up(tiles * sizeof(int), 256);
    b += align_up(tiles * sizeof(float), 256);
    if (with_partials) b += align_up((tiles + fixup_blocks_for(static_cast<int>(tiles))) * 3 * sizeof(double), 256);
    return b + 256;
}

MergePlan merge_plan_carve(void* block, int rows, int nnz, bool with_partials, int ipt) {
    MergePlan p;
    p.ipt = ipt;
    p.num_tiles = merge_num_tiles(rows, nnz, ipt);
    p.fixup_blocks = fixup_blocks_for(p.num_tiles);
    const size_t tiles = static_cast<size_t>(p.num_tiles);
    unsigned char* at = static_cast<unsigned char*>(block);
    p.coords = reinterpret_cast<int2*>(at);
    at += align_up((tiles + 1) * sizeof(int2), 256);
    p.carry_row = reinterpret_cast<int*>(at);
    at += align_up(tiles * sizeof(int), 256);
    p.carry_val = reinterpret_cast<float*>(at);
    at += align_up(tiles * sizeof(float), 256);
    p.partials = with_partials ? reinterpret_cast<double*>(at) : nullptr;
    return p;
}

namespace {

__global__ void merge_partition_kernel(int rows, int nnz, const int* __restrict__ row_ptrs,
                                       int num_tiles, int tile_items, int2* __restrict__ coords) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > num_tiles) return;
    const long long total = static_cast<long long>(rows) + nnz;
    const long long d = static_cast<long long>(t) * tile_items;
    coords[t] = diagonal_search_global(static_cast<int>(d < total ? d : total), row_ptrs, rows, nnz);
}

// block-wide sum of RankSums into partials[slot*3 .. +3] (fixed order)
__device__ __forceinline__ void block_store_sums(const RankSums& s, double* __restrict__ partials, int slot,
                                                 double (*scratch)[3]) {
    double a = dev::warp_sum(s.l2), b = dev::warp_sum(s.l1), c = dev::warp_sum(s.dangling);
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { scratch[warp][0] = a; scratch[warp][1] = b; scratch[warp][2] = c; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < kT / 32; ++w) t += scratch[w][threadIdx.x];
        partials[static_cast<size_t>(slot) * 3 + threadIdx.x] = t;
    }
}
__device__ __forceinline__ void block_store_sums(const NoSums&, double*, int, double (*)[3]) {}

// ---------------------------------------------------------------- level 2 ----

template <class Row, int IPT>
__global__ void __launch_bounds__(kT)
merge_tile_kernel(int rows, int nnz, const int* __restrict__ row_ptrs,
                  const int* __restrict__ col_indices, const float* __restrict__ values,
                  const float* __restrict__ x, const int2* __restrict__ coords,
                  int* __restrict__ carry_row, float* __restrict__ carry_val, Row row_op,
                  double* __restrict__ partials, int use_tma) {
    constexpr int kIPT = IPT;          // shadow the file-level geometry: this kernel's tile is kT * IPT items
    constexpr int kTile = kT * IPT;
    __shared__ __align__(16) int s_end_raw[kTile + 8];  // global END offset of tile-local row i (+ alignment shift)
    __shared__ __align__(16) float s_prod[kTile + 4];   // values, then products in place
    extern __shared__ __align__(16) int s_col[];        // [kTile + 4], allocated for the TMA path only
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ float s_warp_val[kT / 32];
    __shared__ int s_warp_flag[kT / 32];
    __shared__ double s_sums[kT / 32][3];

    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const int2 c0 = coords[tile];
    const int2 c1 = coords[tile + 1];
    const int row_s = c0.x, nz_s = c0.y;
    const int tile_rows = c1.x - c0.x;  // row-end items in this tile
    const int tile_nz = c1.y - c0.y;    // non-zero items in this tile
    const int tile_items = tile_rows + tile_nz;
    const int nz_e = c1.y;

    const float row_ctx = row_op.prepare();

    const int base = nz_s & ~3;
    const bool vec_ok = dev::aligned16(values) && dev::aligned16(col_indices);  // any device pointer is legal

    // ---- TMA path: three 1-D bulk copies (row ends, values, col_indices of the tile) onto one
    // mbarrier; the stream bypasses registers and L1, which on scale-free inputs is the unit that
    // saturates (one L1 wavefront per gathered x element).  Needs 16-byte aligned arrays and spans
    // that stay inside them, i.e. every tile except the last one or two.
    const int end_first = (row_s + 1) & ~3;                         // aligned start of the row-end span
    const int end_count = ((row_s + 1 + tile_rows + 1 + 3) & ~3) - end_first;
    const int nz_end4 = (nz_e + 3) & ~3;
    auto gather = [&](int c) { return dev::ld_x(x + c); };  // L1-allocating: hub columns hit (no_allocate measured slower)
    const bool tma_ok = use_tma && vec_ok && dev::aligned16(row_ptrs) && (c1.x < rows) &&
                        (end_first + end_count <= rows + 1) && (nz_end4 <= (nnz & ~3)) && (nz_e > nz_s);
    const int* s_end = s_end_raw + (tma_ok ? (row_s + 1 - end_first) : 0);
    if (tma_ok) {
        if (tid == 0) {
            dev::mbar_init(&s_bar, 1);
            dev::mbar_fence_init();
        }
        __syncthreads();
        if (tid == 0) {
            const uint32_t nz_bytes = static_cast<uint32_t>(nz_end4 - base) * 4u;
            const uint32_t end_bytes = static_cast<uint32_t>(end_count) * 4u;
            dev::mbar_arrive_expect_tx(&s_bar, 2u * nz_bytes + end_bytes);
            dev::tma_bulk_g2s(s_end_raw, row_ptrs + end_first, end_bytes, &s_bar);
            dev::tma_bulk_g2s(s_prod, values + base, nz_bytes, &s_bar);
            dev::tma_bulk_g2s(s_col, col_indices + base, nz_bytes, &s_bar);
        }
        dev::mbar_wait(&s_bar, 0);
        // products in place: all gathers of a thread are issued before the first multiply
        constexpr int kPer = (kTile + kT - 1) / kT;
        float xv[kPer];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int j = nz_s + tid + u * kT;
            if (j < nz_e) xv[u] = gather(s_col[j - base]);
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int j = nz_s + tid + u * kT;
            if (j < nz_e) s_prod[j - base] *= xv[u];
        }
    } else {
    // ---- stage row ends (tile_rows + 1 entries; the last one bounds the open row)
    for (int i = tid; i <= tile_rows; i += kT)
        s_end_raw[i] = (row_s + i < rows) ? dev::ld_stream_i(row_ptrs + row_s + 1 + i) : INT_MAX;

    // ---- stage products of non-zeros [nz_s, nz_e) at slot (j - base) ----------
    for (int j = base + 4 * tid; j < nz_e; j += 4 * kT) {
        float p0, p1, p2, p3;
        if (vec_ok && j >= nz_s && j + 4 <= nz_e) {
            const float4 v = dev::ld_stream_f4(values + j);
            const int4 c = dev::ld_stream_i4(col_indices + j);
            p0 = v.x * gather(c.x);
            p1 = v.y * gather(c.y);
            p2 = v.z * gather(c.z);
            p3 = v.w * gather(c.w);
        } else {
            p0 = (j + 0 >= nz_s && j + 0 < nz_e) ? values[j + 0] * gather(col_indices[j + 0]) : 0.0f;
            p1 = (j + 1 >= nz_s && j + 1 < nz_e) ? values[j + 1] * gather(col_indices[j + 1]) : 0.0f;
            p2 = (j + 2 >= nz_s && j + 2 < nz_e) ? values[j + 2] * gather(col_indices[j + 2]) : 0.0f;
            p3 = (j + 3 >= nz_s && j + 3 < nz_e) ? values[j + 3] * gather(col_indices[j + 3]) : 0.0f;
        }
        *reinterpret_cast<float4*>(s_prod + (j - base)) = make_float4(p0, p1, p2, p3);
    }
    }  // register-staged path
    // does the tile's first row own non-zeros in earlier tiles?
    const bool first_row_split = (row_s < rows) && (nz_s > __ldg(row_ptrs + row_s));
    __syncthreads();

    // ---- per-thread diagonal inside the tile (search in shared memory) ---------
    const int diag = min(tid * kIPT, tile_items);
    int lo = max(diag - tile_nz, 0);
    int hi = min(diag, tile_rows);
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (s_end[mid] <= nz_s + (diag - mid - 1)) lo = mid + 1;
        else hi = mid;
    }
    int r = lo;                  // tile-local row
    int z = nz_s + (diag - lo);  // global non-zero index
    const int my_items = min(kIPT, tile_items - diag);

    typename Row::Sums sums;
    sums.clear();

    float running = 0.0f;
    bool emitted = false;
    float first_sum = 0.0f;
    int first_row = 0;
    int row_end = s_end[r];
#pragma unroll
    for (int it = 0; it < kIPT; ++it) {
        if (it < my_items) {
            if (z < row_end) {
                running += s_prod[z - base];
                ++z;
            } else {
                if (!emitted) {  // may still need the carry of earlier threads
                    emitted = true;
                    first_sum = running;
                    first_row = r;
                } else {
                    row_op.tile_finish(row_s + r, running, sums, row_ctx);
                }
                running = 0.0f;
                ++r;
                row_end = s_end[r];
            }
        }
    }

    // ---- segmented scan of (emitted, running) over the CTA ----------------------
    // combine(earlier, later) = (fe | fl, fl ? vl : ve + vl)
    const int lane = tid & 31, warp = tid >> 5;
    float v = running;
    int f, ex_f;
    float ex_v;
    warp_segmented_scan(v, emitted, lane, f, ex_v, ex_f);
    if (lane == 31) { s_warp_val[warp] = v; s_warp_flag[warp] = f; }
    __syncthreads();
    // fold the aggregates of the preceding warps
    float pre_v = 0.0f;
    int pre_f = 0;
    for (int w = 0; w < warp; ++w) {
        const float wv = s_warp_val[w];
        const int wf = s_warp_flag[w];
        pre_v = wf ? wv : pre_v + wv;
        pre_f |= wf;
    }
    const float carry_in = ex_f ? ex_v : pre_v + ex_v;

    if (emitted) {
        const float total = carry_in + first_sum;
        if (first_row == 0 && first_row_split) row_op.park(row_s, total);  // level 3 finishes it
        else row_op.tile_finish(row_s + first_row, total, sums, row_ctx);
    }

    // ---- tile carry-out: the row still open at the tile end ------------------------
    if (tid == kT - 1) {
        const float open_sum = f ? v : pre_v + v;  // inclusive scan value of the last thread
        const int row_e = c1.x;
        const int open_start = tile_rows > 0 ? s_end[tile_rows - 1] : (row_s < rows ? __ldg(row_ptrs + row_s) : nz_e);
        const bool has_open = (row_e < rows) && (nz_e > max(open_start, nz_s));
        carry_row[tile] = has_open ? row_e : -1;
        carry_val[tile] = has_open ? open_sum : 0.0f;
    }

    if (Row::kReduces) {
        __syncthreads();  // every raw row sum of this CTA is visible CTA-wide
        row_op.tile_epilogue(row_s + (first_row_split ? 1 : 0), c1.x, tid, sums, row_ctx);
        block_store_sums(sums, partials, tile, s_sums);
    }
}

// ---------------------------------------------------------------- level 3 ----

template <class Row>
__global__ void __launch_bounds__(256)
merge_fixup_kernel(int num_tiles, const int* __restrict__ carry_row, const float* __restrict__ carry_val,
                   Row row_op, double* __restrict__ partials, int partial_base) {
    __shared__ double s_sums[256 / 32][3];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    typename Row::Sums sums;
    sums.clear();
    const float row_ctx = row_op.prepare();
    if (t < num_tiles) {
        const int row = carry_row[t];
        if (row >= 0 && (t == 0 || carry_row[t - 1] != row)) {  // leader of a run of tiles
            float total = carry_val[t];
            for (int u = t + 1; u < num_tiles && carry_row[u] == row; ++u) total += carry_val[u];
            // the tile in which the row ends parked its own share
            row_op.finish(row, row_op.parked(row) + total, sums, row_ctx);
            row_op.publish_row(row);
        }
    }
    if (Row::kReduces) block_store_sums(sums, partials, partial_base + blockIdx.x, s_sums);
}

// final deterministic reduction of the per-CTA partial sums -> out[3]
__global__ void __launch_bounds__(1024)
reduce_partials_kernel(const double* __restrict__ partials, int count, double* __restrict__ out) {
    __shared__ double s[32][3];
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = threadIdx.x; i < count; i += 1024) {
        a += partials[static_cast<size_t>(i) * 3 + 0];
        b += partials[static_cast<size_t>(i) * 3 + 1];
        c += partials[static_cast<size_t>(i) * 3 + 2];
    }
    a = dev::warp_sum(a); b = dev::warp_sum(b); c = dev::warp_sum(c);
    if ((threadIdx.x & 31) == 0) { s[threadIdx.x >> 5][0] = a; s[threadIdx.x >> 5][1] = b; s[threadIdx.x >> 5][2] = c; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += s[w][threadIdx.x];
        out[threadIdx.x] = t;
    }
}

template <class Row>
cudaError_t run_tiles(const CsrView& A, const float* x, const MergePlan& plan, const Row& row_op,
                      cudaStream_t stream) {
    if (plan.num_tiles <= 0) return cudaSuccess;
    static const int use_tma = env_int("SPMV_B200_MERGE_TMA", 0);
    static const int carveout = env_int("SPMV_B200_MERGE_CARVEOUT", -1);
    auto launch = [&](auto kernel, int ipt) {
        if (carveout >= 0) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
        const size_t dyn_smem = use_tma ? (kT * ipt + 4) * sizeof(int) : 0;
        kernel<<<plan.num_tiles, kT, dyn_smem, stream>>>(A.rows, A.nnz, A.row_ptrs, A.col_indices, A.values, x, plan.coords,
                                                         plan.carry_row, plan.carry_val, row_op, plan.partials, use_tma);
    };
    if (plan.ipt == 8) launch(merge_tile_kernel<Row, 8>, 8);
    else if (plan.ipt == kMergeItemsPerThread) launch(merge_tile_kernel<Row, kMergeItemsPerThread>, kMergeItemsPerThread);
    else return cudaErrorInvalidValue;
    merge_fixup_kernel<Row><<<plan.fixup_blocks, 256, 0, stream>>>(plan.num_tiles, plan.carry_row, plan.carry_val,
                                                                   row_op, plan.partials, plan.num_tiles);
    count_launches(2);
    return cudaGetLastError();
}

}  // namespace

int merge_items_for(int rows, int nnz) {
    static const int forced = env_int("SPMV_B200_MERGE_IPT", 0);  // 7 / 8: A/B timing
    if (forced == 7 || forced == 8) return forced;
    // measured (scripts/time_mid.py, bench_hot.py; 7 / 8 items): config 2 0.380 / 0.321 ms, 7-point stencil
    // 0.129 / 0.102, 9-point 0.154 / 0.134, random rows avg 5 and 8 equal, avg 12-24 0.271 / 0.273 .. 0.488 / 0.498,
    // config 3 (avg 3) 2.19 / 2.27, R-MAT 24 (avg 16) 1.27 / 1.37 -> 8 items for 4 <= avg < 10 only
    const double avg = rows > 0 ? static_cast<double>(nnz) / rows : 0.0;
    return (avg >= 4.0 && avg < 10.0) ? 8 : kMergeItemsPerThread;
}

cudaError_t launch_merge_partition(const CsrView& A, const MergePlan& plan, cudaStream_t stream) {
    if (plan.num_tiles <= 0) return cudaSuccess;
    const int n = plan.num_tiles + 1;
    merge_partition_kernel<<<(n + 255) / 256, 256, 0, stream>>>(A.rows, A.nnz, A.row_ptrs, plan.num_tiles, kT * plan.ipt,
                                                                plan.coords);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_merge_spmv(const CsrView& A, const float* x, float* y, const MergePlan& plan,
                              cudaStream_t stream) {
    if (A.rows <= 0) return cudaSuccess;
    PlainRow op{y};
    return run_tiles(A, x, plan, op, stream);
}

// Level 3 alone, for tile kernels that live elsewhere (csr_hot_kernels.cu).  The PageRank flavour
// also folds the `partial_base` per-worker sums written by the tile kernel and its own per-CTA sums.
cudaError_t launch_merge_fixup(const MergePlan& plan, float* y, cudaStream_t stream) {
    if (plan.num_tiles <= 0) return cudaSuccess;
    PlainRow op{y};
    merge_fixup_kernel<PlainRow><<<plan.fixup_blocks, 256, 0, stream>>>(plan.num_tiles, plan.carry_row, plan.carry_val,
                                                                        op, plan.partials, 0);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_merge_fixup_pagerank(const MergePlan& plan, const PageRankStepArgs& args, int partial_base,
                                        cudaStream_t stream) {
    if (plan.num_tiles <= 0) return cudaSuccess;
    PageRankRow op{args};
    merge_fixup_kernel<PageRankRow><<<plan.fixup_blocks, 256, 0, stream>>>(plan.num_tiles, plan.carry_row,
                                                                           plan.carry_val, op, plan.partials, partial_base);
    reduce_partials_kernel<<<1, 1024, 0, stream>>>(plan.partials, partial_base + plan.fixup_blocks, args.out);
    count_launches(2);
    return cudaGetLastError();
}

cudaError_t launch_reduce_partials(const double* partials, int count, double* out, cudaStream_t stream) {
    reduce_partials_kernel<<<1, 1024, 0, stream>>>(partials, count, out);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_merge_pagerank(const CsrView& A, const MergePlan& plan, const PageRankStepArgs& args,
                                  cudaStream_t stream) {
    if (A.rows <= 0) {
        cudaError_t e = cudaMemsetAsync(args.out, 0, 3 * sizeof(double), stream);
        return e;
    }
    PageRankRow op{args};
    cudaError_t e = run_tiles(A, args.r_old, plan, op, stream);
    if (e != cudaSuccess) return e;
    reduce_partials_kernel<<<1, 1024, 0, stream>>>(plan.partials, plan.num_tiles + plan.fixup_blocks, args.out);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace b200
}  // namespace spmv
