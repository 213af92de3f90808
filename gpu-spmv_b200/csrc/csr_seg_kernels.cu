// csr_seg_kernels.cu -- planned CSR SpMV as a register-resident segmented reduction
// ("segmented stream").  One of the two kernels behind CSR plans (spmv_b200_csr_plan and the
// automatic plans of spmv_csr(MERGE_PATH)): planned_build() (dispatch.cu) picks it for matrices
// WITHOUT hub columns and with >= 4 non-zeros per row; scale-free matrices and PageRank shards
// take the hub-column merge-path kernel (csr_hot_kernels.cu).  It replaces the same reference code
// as the merge-path kernels (src/spmv_kernels.cu:48-130,267) for callers that multiply by the same
// sparsity pattern more than once.
//
// Idea.  ncu (profiles/r1_hub_kernel.md): the merge-path tile kernels are bound by the L1TEX data
// pipe, and a third of their wavefronts on it are the algorithm's own shared-memory traffic
// (products parked in shared memory, a binary search per thread, row ends re-read in the consume
// loop).  A plan may hold a private re-encoding of col_indices, so the row structure can travel
// WITH the stream instead of being searched for:
//
//   enc[j]  bit 31  the column is a hub: bits 0..29 = slot of the shared-memory x table
//           bit 30  non-zero j is the FIRST of its row ("head")
//           else    bits 0..29 = column
//   rows_nz[k]          row of the k-th head (rows without non-zeros never appear)
//   span_head_base[s]   number of heads before non-zero s * 256 (one entry per warp and tile)
//
// A tile is 2048 consecutive non-zeros of one 256-thread worker (4 workers per persistent
// 1024-thread CTA, one CTA per SM, as in csr_hot_kernels.cu).  A lane owns two runs of 4
// consecutive non-zeros (two 128-bit loads of values and of enc, fully coalesced), gathers its 8 x
// entries (hub columns from the table), and reduces its runs serially IN REGISTERS: sums closed
// inside a run are stored straight to y[rows_nz[.]]; the open ends are combined by a warp-shuffle
// segmented scan whose flags come from one ballot (only values are shuffled), then across the 8
// warps through a few words of shared memory, then across tiles by a fix-up kernel (tile_lead /
// tile_tail), always in index order -- deterministic, no atomics.  No search, no products in
// shared memory, no row_ptrs traffic, no merge items for empty rows.  Rows without non-zeros are
// never touched: y is zeroed first (plain SpMV) or the PageRank epilogue kernel substitutes 0 (bit
// mask of non-empty rows).  scripts/seg_model.py is an executable model of the index logic.
//
// Measured (profiles/r1_hub_kernel.md): Laplacian 4096^2 0.263 ms against 0.382 ms for merge-path
// (3.3 TB/s, 51 % of the measured HBM peak); R-MAT 24 1.12 ms against 1.04 ms for the hub-column
// kernel -- warp shuffles occupy the same data pipe as shared-memory accesses, and the instruction
// count equals merge-path's, so on a gather-bound matrix the shorter critical path of merge-path's
// 4 overlapping workers wins.  Its PageRank form exchanges the slices in a separate epilogue pass
// (no overlap with the product), which costs 25 % on 8 GPUs; PageRank plans do not use it.
//
// Roofline: HBM; algorithmic bytes as for every CSR kernel (8*nnz + 4*(rows+1) + 4*cols
// + 4*rows, reference src/bandwidth.cpp:34-42).  The kernel reads 8 B per non-zero + 4 B per
// non-empty row + 4 B per 256 non-zeros + x, and writes y.
#include "device_utils.cuh"
#include "internal.hpp"

#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

namespace spmv {
namespace b200 {
namespace {

constexpr int kWorkers = 4;
constexpr int kWT = 256;                      // threads per worker
constexpr int kThreads = kWorkers * kWT;      // 1024
constexpr int kWarps = kWT / 32;              // warps per worker
constexpr int kRun = 4;                       // consecutive non-zeros per lane and step
constexpr int kSteps = 2;                     // steps per tile
constexpr int kWarpSpan = 32 * kRun * kSteps; // 256 non-zeros per warp and tile
constexpr int kTile = kSegTile;
static_assert(kTile == kWarps * kWarpSpan, "tile geometry");
constexpr unsigned kHotBit = 0x80000000u;
constexpr unsigned kHeadBit = 0x40000000u;
constexpr unsigned kIdxMask = 0x3fffffffu;
constexpr int kBlock = 256;

__device__ __forceinline__ void worker_sync(int w) {
    asm volatile("bar.sync %0, %1;" :: "r"(w + 1), "n"(kWT) : "memory");
}

// x entry of an encoded column (predicated: a lane that reads the table issues no L1 wavefront)
__device__ __forceinline__ float gather_enc(int e, uint32_t s_hot_addr, const float* __restrict__ x) {
    float r;
    const uint32_t idx = static_cast<uint32_t>(e) & kIdxMask;
    const uint32_t sa = s_hot_addr + (idx << 2);
    const unsigned long long ga = reinterpret_cast<unsigned long long>(x) + (static_cast<unsigned long long>(idx) << 2);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.lt.s32 p, %1, 0;\n"
        "@p ld.shared.f32 %0, [%2];\n"
        "@!p ld.global.nc.f32 %0, [%3];\n"
        "}\n"
        : "=f"(r)
        : "r"(e), "r"(sa), "l"(ga));
    return r;
}

struct Stream {  // one tile's share of a lane: two runs of four
    float4 v[kSteps];
    int4 e[kSteps];
};

__device__ __forceinline__ void load_stream(Stream& s, int j_first, int nnz, bool vec_ok, const float* __restrict__ values,
                                            const int* __restrict__ enc) {
#pragma unroll
    for (int c = 0; c < kSteps; ++c) {
        const int j = j_first + c * 32 * kRun;
        s.e[c] = dev::ld_stream_i4(enc + j);  // enc is padded to whole tiles
        if (vec_ok && j + kRun <= nnz) {
            s.v[c] = dev::ld_stream_f4(values + j);
        } else {  // array tail or an unaligned values pointer
            s.v[c].x = j + 0 < nnz ? dev::ld_stream_f(values + j + 0) : 0.0f;
            s.v[c].y = j + 1 < nnz ? dev::ld_stream_f(values + j + 1) : 0.0f;
            s.v[c].z = j + 2 < nnz ? dev::ld_stream_f(values + j + 2) : 0.0f;
            s.v[c].w = j + 3 < nnz ? dev::ld_stream_f(values + j + 3) : 0.0f;
        }
    }
}

__device__ __forceinline__ int head_bits(const int4& e) {
    return ((e.x >> 30) & 1) | (((e.y >> 30) & 1) << 1) | (((e.z >> 30) & 1) << 2) | (((e.w >> 30) & 1) << 3);
}

// Shared memory: [x table: hot_slots floats][kWorkers x 2 (tile parity) x {flag[8] int, lead[8] float, tail[8] float, 8 spare}]
constexpr size_t kSegFixedSmem = kWorkers * kWarps * 32;

__global__ void __launch_bounds__(kThreads, 1)
seg_spmv_kernel(int nnz, const int* __restrict__ enc, const float* __restrict__ values, const float* __restrict__ x,
                const int* __restrict__ hot_cols, int n_hot, const int* __restrict__ rows_nz,
                const int* __restrict__ span_head_base, int num_tiles, float* __restrict__ y,
                float* __restrict__ tile_lead, float* __restrict__ tile_tail) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int hot_slots = (n_hot + 3) & ~3;
    float* s_hot = reinterpret_cast<float*>(smem_raw);
    const int tid = threadIdx.x;
    const int w = tid / kWT;
    const int wt = tid % kWT;
    const int lane = wt & 31, warp = wt >> 5;
    int* s_fold = reinterpret_cast<int*>(s_hot + hot_slots) + w * 8 * kWarps;  // [parity][flag, lead, tail, spare][warp]

    // ---- the table: x of the hub columns (all of x when hot_cols == nullptr), once per CTA ----
    for (int i = tid; i < hot_slots; i += kThreads)
        s_hot[i] = i < n_hot ? dev::ld_x(x + (hot_cols ? __ldg(hot_cols + i) : i)) : 0.0f;
    __syncthreads();
    const uint32_t s_hot_addr = dev::smem_u32(s_hot);
    const bool vec_ok = dev::aligned16(values);
    const unsigned lt_mask = (1u << lane) - 1u;

    const int stride = gridDim.x * kWorkers;
    int tile = w * gridDim.x + blockIdx.x;
    Stream cur;
    int shb = 0;  // heads before this warp's span (from the plan: no barrier, no counting pass)
    if (tile < num_tiles) {
        load_stream(cur, tile * kTile + warp * kWarpSpan + lane * kRun, nnz, vec_ok, values, enc);
        shb = __ldg(span_head_base + tile * kWarps + warp);
    }

    int parity = 0;
    while (tile < num_tiles) {
        const int next = tile + stride;
        const int j_first = tile * kTile + warp * kWarpSpan + lane * kRun;
        int* s_flag = s_fold + parity * 4 * kWarps;
        float* s_lead = reinterpret_cast<float*>(s_flag + kWarps);
        float* s_tail = s_lead + kWarps;
        int shb_next = 0;
        if (next < num_tiles) shb_next = __ldg(span_head_base + next * kWarps + warp);

        // ---- x gathers: all 8 issued before anything waits on them -----------------------
        float p[kSteps][kRun];
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
            p[c][0] = gather_enc(cur.e[c].x, s_hot_addr, x);
            p[c][1] = gather_enc(cur.e[c].y, s_hot_addr, x);
            p[c][2] = gather_enc(cur.e[c].z, s_hot_addr, x);
            p[c][3] = gather_enc(cur.e[c].w, s_hot_addr, x);
        }

        // ---- next tile's stream: issued right behind the gathers, so its DRAM latency overlaps theirs ----
        Stream nxt;
        if (next < num_tiles) load_stream(nxt, next * kTile + warp * kWarpSpan + lane * kRun, nnz, vec_ok, values, enc);

        // ---- head bookkeeping (needs enc only, so it overlaps the gathers) ------------------
        int hbits[kSteps];
        unsigned head_lanes[kSteps];  // lanes whose run holds a head
        int before[kSteps];           // heads of this span before this lane's run
        int span_heads = 0;
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
            hbits[c] = head_bits(cur.e[c]);
            const int n = __popc(hbits[c]);
            const unsigned b0 = __ballot_sync(0xffffffffu, n & 1);
            const unsigned b1 = __ballot_sync(0xffffffffu, n & 2);
            const unsigned b2 = __ballot_sync(0xffffffffu, n & 4);
            head_lanes[c] = b0 | b1 | b2;
            before[c] = span_heads + __popc(b0 & lt_mask) + 2 * __popc(b1 & lt_mask) + 4 * __popc(b2 & lt_mask);
            span_heads += __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
        }
        // row of the segment a run closes most often, the one ended by its first head (segments that
        // start AND end inside a run of 4 are rarer; their rows are fetched when they occur)
        int row_a[kSteps];
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
            const int hb = shb + before[c];
            row_a[c] = (hbits[c] != 0 && hb >= 1) ? __ldg(rows_nz + hb - 1) : -1;
        }
        int lead_row = -1;  // lane 0: the row open at the start of this warp's span
        if (lane == 0 && span_heads > 0 && shb >= 1) lead_row = __ldg(rows_nz + shb - 1);

        // ---- products (non-zeros past the end of the matrix contribute an exact 0) ------------
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
            const int j = j_first + c * 32 * kRun;
            p[c][0] = j + 0 < nnz ? cur.v[c].x * p[c][0] : 0.0f;
            p[c][1] = j + 1 < nnz ? cur.v[c].y * p[c][1] : 0.0f;
            p[c][2] = j + 2 < nnz ? cur.v[c].z * p[c][2] : 0.0f;
            p[c][3] = j + 3 < nnz ? cur.v[c].w * p[c][3] : 0.0f;
        }
        cur = nxt;

        // ---- the two steps of this warp, in non-zero order --------------------------------------
        float open_sum = 0.0f;   // sum of the segment open at the current position (warp-uniform)
        bool seen = false;       // a head has been passed in this warp's span (warp-uniform)
        float warp_lead = 0.0f;  // sum of the span before its first head (valid on one lane)
        bool has_lead = false;
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
            // serial walk of the run
            float acc = 0.0f, lead = 0.0f, closed0 = 0.0f, closed1 = 0.0f, closed2 = 0.0f;
            int n = 0;
#pragma unroll
            for (int k = 0; k < kRun; ++k) {
                if ((hbits[c] >> k) & 1) {
                    if (n == 0) lead = acc;
                    else if (n == 1) closed0 = acc;
                    else if (n == 2) closed1 = acc;
                    else closed2 = acc;
                    ++n;
                    acc = 0.0f;
                }
                acc += p[c][k];
            }
            // Segmented inclusive scan of the tails over the lanes.  Before the level of distance d
            // a lane holds the sum of the window (lane - d, lane] cut at the nearest head; whether
            // that window holds a head is read off the ballot, so only the values are shuffled.
            const unsigned m = head_lanes[c];
            float v = acc;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float pv = __shfl_up_sync(0xffffffffu, v, d);
                const unsigned window = ((2u << lane) - 1u) & ~((lane >= d ? (2u << (lane - d)) : 1u) - 1u);  // lanes (lane-d, lane]
                if (lane >= d && !(m & window)) v = pv + v;
            }
            float ex_v = __shfl_up_sync(0xffffffffu, v, 1);
            if (lane == 0) ex_v = 0.0f;
            const bool ex_f = (m & lt_mask) != 0;  // a head in an earlier lane of this step
            const float carry_in = ex_f ? ex_v : open_sum + ex_v;
            if (n > 0) {
                const float total = carry_in + lead;  // the segment ended by this lane's first head
                if (ex_f || seen) {
                    y[row_a[c]] = total;
                } else {  // it started before this warp's span: resolved after the cross-warp fold
                    warp_lead = total;
                    has_lead = true;
                }
                if (n > 1) {
                    const int hb = shb + before[c];
                    y[__ldg(rows_nz + hb)] = closed0;
                    if (n > 2) y[__ldg(rows_nz + hb + 1)] = closed1;
                    if (n > 3) y[__ldg(rows_nz + hb + 2)] = closed2;
                }
            }
            const float v31 = __shfl_sync(0xffffffffu, v, 31);
            open_sum = m ? v31 : open_sum + v31;
            seen = seen || m != 0;
        }
        const unsigned lead_mask = __ballot_sync(0xffffffffu, has_lead);
        if (lead_mask) warp_lead = __shfl_sync(0xffffffffu, warp_lead, __ffs(lead_mask) - 1);
        if (lane == 0) {
            s_flag[warp] = seen ? 1 : 0;
            s_lead[warp] = warp_lead;
            s_tail[warp] = open_sum;
        }
        worker_sync(w);

        // ---- across the warps of the tile (index order) ------------------------------------------
        if (lane == 0) {
            float carry = 0.0f;
            bool has = false;
            for (int k = 0; k < warp; ++k) {
                const int fk = s_flag[k];
                const float tk = s_tail[k];
                carry = fk ? tk : carry + tk;
                has = has || fk;
            }
            if (seen) {
                const float total = carry + warp_lead;
                if (has) y[lead_row] = total;
                else tile_lead[tile] = total;  // the segment open at the start of the tile
                carry = open_sum;
                has = true;
            } else {
                carry += open_sum;
            }
            if (warp == kWarps - 1) {
                tile_tail[tile] = carry;  // the segment open at the end of the tile (whole tile if no head)
                if (!has) tile_lead[tile] = 0.0f;
            }
        }
        // The fold slots alternate with the tile parity: a warp reaches the slots of this parity again
        // only after the NEXT tile's barrier, which every folding lane 0 of this tile must reach first.
        parity ^= 1;
        tile = next;
        shb = shb_next;
    }
}

// The segment open at the end of every tile that holds a head: its tail, the whole sums of the
// head-less tiles that follow and the lead of the next tile with a head, in tile order.
__global__ void __launch_bounds__(kBlock)
seg_fixup_kernel(int num_tiles, const int* __restrict__ span_head_base, const int* __restrict__ rows_nz,
                 const float* __restrict__ tile_lead, const float* __restrict__ tile_tail, float* __restrict__ y) {
    const int t = blockIdx.x * kBlock + threadIdx.x;
    if (t >= num_tiles) return;
    auto tile_head_base = [&](int tile) { return __ldg(span_head_base + static_cast<size_t>(tile) * kWarps); };
    const int last_head = tile_head_base(t + 1) - 1;
    if (last_head < tile_head_base(t)) return;  // no head in this tile
    float total = tile_tail[t];
    int u = t + 1;
    while (u < num_tiles && tile_head_base(u + 1) == tile_head_base(u)) total += tile_tail[u++];
    if (u < num_tiles) total += tile_lead[u];
    y[rows_nz[last_head]] = total;
}

// PageRank update of every row of the shard from the raw sums left in r_new (rows without
// non-zeros were never written: their sum is 0), residuals and next dangling mass, and the copy
// of the finished values into the peers' vectors (fused slice exchange).  The update is
// dev::pr_row_value, as in PageRankRowT::finish.
__global__ void __launch_bounds__(kBlock)
seg_pagerank_epilogue_kernel(PageRankStepArgs a, int rows, const uint32_t* __restrict__ nonempty,
                             double* __restrict__ partials) {
    __shared__ double s_sums[kBlock / 32][3];
    const float dangling_term = dev::pr_step_context(a.damping, *a.d_dsum, a.n_global, a.pvec);
    double l2 = 0.0, l1 = 0.0, dangling = 0.0;
    for (long long i = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; i < rows;
         i += static_cast<long long>(gridDim.x) * kBlock) {
        const int g = a.row_offset + static_cast<int>(i);
        const float raw = ((nonempty[i >> 5] >> (i & 31)) & 1u) ? a.r_new[g] : 0.0f;
        const float v = dev::pr_row_value(a.damping, raw, dangling_term, a.teleport, a.pvec, static_cast<int>(i));
        a.r_new[g] = v;
        const double diff = static_cast<double>(v) - static_cast<double>(a.r_old[g]);
        l2 += diff * diff;
        l1 += fabs(diff);
        if ((a.bits[g >> 5] >> (g & 31)) & 1u) dangling += static_cast<double>(v);
        if (a.n_peers > 1) {
            if (a.mc_r_new) {
                dev::st_multicast_f(a.mc_r_new + g, v);  // NVSwitch multicast: one store reaches every peer
            } else {
#pragma unroll
                for (int p = 0; p < kMaxPeers; ++p)  // static indices: the pointer table stays in the constant bank
                    if (p < a.n_peers && p != a.self_rank) a.peers[p][g] = v;
            }
        }
    }
    l2 = dev::warp_sum(l2); l1 = dev::warp_sum(l1); dangling = dev::warp_sum(dangling);
    if ((threadIdx.x & 31) == 0) { s_sums[threadIdx.x >> 5][0] = l2; s_sums[threadIdx.x >> 5][1] = l1; s_sums[threadIdx.x >> 5][2] = dangling; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int k = 0; k < kBlock / 32; ++k) t += s_sums[k][threadIdx.x];
        partials[static_cast<size_t>(blockIdx.x) * 3 + threadIdx.x] = t;
    }
}

// ---------------------------------------------------------------------------- plan kernels ----

inline unsigned plan_grid(long long n) {
    long long b = (n + kBlock - 1) / kBlock;
    if (b < 1) b = 1;
    return static_cast<unsigned>(b < 148 * 16 ? b : 148 * 16);
}

// enc[j] for j < padded: hub slot / column (no head bits yet); padding reads slot 0
__global__ void seg_encode_kernel(int nnz, int padded, int cols, const int* __restrict__ col_indices,
                                  const int* __restrict__ slot_of, int* __restrict__ enc) {
    for (long long j = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; j < padded;
         j += static_cast<long long>(gridDim.x) * kBlock) {
        unsigned e = kHotBit;  // slot 0
        if (j < nnz) {
            const int c = dev::ld_stream_i(col_indices + j);
            if (c >= 0 && c < cols) {
                if (!slot_of) e = kHotBit | static_cast<unsigned>(c);  // the table is x itself
                else {
                    const int s = __ldg(slot_of + c);
                    e = s >= 0 ? (kHotBit | static_cast<unsigned>(s)) : static_cast<unsigned>(c);
                }
            }
        }
        enc[j] = static_cast<int>(e);
    }
}

// marks the first non-zero of every non-empty row, flags[r] = row r has non-zeros, and the same as a bit mask
__global__ void seg_heads_kernel(int rows, const int* __restrict__ row_ptrs, int* __restrict__ enc,
                                 unsigned char* __restrict__ flags, uint32_t* __restrict__ nonempty) {
    const int rows_up = (rows + 31) & ~31;
    for (long long r = blockIdx.x * static_cast<long long>(kBlock) + threadIdx.x; r < rows_up;
         r += static_cast<long long>(gridDim.x) * kBlock) {
        bool ne = false;
        if (r < rows) {
            const int a = row_ptrs[r], b = row_ptrs[r + 1];
            ne = b > a;
            flags[r] = ne ? 1 : 0;
            if (ne) enc[a] |= static_cast<int>(kHeadBit);
        }
        const unsigned m = __ballot_sync(0xffffffffu, ne);
        if ((threadIdx.x & 31) == 0) nonempty[r >> 5] = m;
    }
}

// span_head_base[s] = number of non-empty rows that start before non-zero s * kWarpSpan
// (s = tile * kWarps + warp; entry num_spans closes the table)
__global__ void seg_span_heads_kernel(int num_spans, int n_heads, const int* __restrict__ row_ptrs,
                                      const int* __restrict__ rows_nz, int* __restrict__ tile_head_base) {
    const int t = blockIdx.x * kBlock + threadIdx.x;
    if (t > num_spans) return;
    const long long target = static_cast<long long>(t) * kWarpSpan;
    int lo = 0, hi = n_heads;
    while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);
        if (__ldg(row_ptrs + __ldg(rows_nz + mid)) < target) lo = mid + 1;
        else hi = mid;
    }
    tile_head_base[t] = lo;
}

cudaError_t run_seg(const SegPlan& P, const float* values, const float* x, float* y, cudaStream_t stream) {
    const size_t smem = static_cast<size_t>((P.n_hot + 3) & ~3) * 4 + kSegFixedSmem;
    cudaError_t e = cudaFuncSetAttribute(seg_spmv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    int grid = device_sm_count();  // persistent: one CTA per SM
    const int want = (P.num_tiles + kWorkers - 1) / kWorkers;
    if (grid > want) grid = want;
    if (grid < 1) grid = 1;
    seg_spmv_kernel<<<grid, kThreads, smem, stream>>>(P.nnz, P.enc, values, x, P.hot_cols, P.n_hot, P.rows_nz,
                                                      P.tile_head_base, P.num_tiles, y, P.tile_lead, P.tile_tail);
    seg_fixup_kernel<<<(P.num_tiles + kBlock - 1) / kBlock, kBlock, 0, stream>>>(P.num_tiles, P.tile_head_base, P.rows_nz,
                                                                               P.tile_lead, P.tile_tail, y);
    count_launches(2);
    return cudaGetLastError();
}

}  // namespace

// ------------------------------------------------------------------------------ host side ----

int seg_table_capacity() {
    int dev_id = 0, optin = 0;
    cudaGetDevice(&dev_id);
    if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev_id) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    const long long room = static_cast<long long>(optin) - static_cast<long long>(kSegFixedSmem) - 64;
    return room > 0 ? static_cast<int>(room / 4) & ~1023 : 0;
}

// Table size used when the caller does not ask for one.  Not the maximum: shared memory is carved
// out of the same 256 KB as the L1, whose lines track the outstanding gather misses.
int seg_default_capacity() {
    static const int env_cap = env_int("SPMV_B200_HOT_CAP", 0);
    const int cap = seg_table_capacity();
    const int want = env_cap > 0 ? (env_cap & ~3) : 24576;
    return want < cap ? want : cap;
}

bool seg_worthwhile(const CsrView& A) {
    // the persistent grid wants a few tiles per worker; below that the one-tile-per-CTA kernels win
    return A.nnz / kTile >= kWorkers * device_sm_count() * 2;
}

void seg_plan_release(SegPlan* p) {
    if (!p) return;
    cudaFree(p->enc); cudaFree(p->hot_cols); cudaFree(p->rows_nz); cudaFree(p->tile_head_base);
    cudaFree(p->nonempty); cudaFree(p->tile_lead); cudaFree(p->tile_tail); cudaFree(p->partials);
    *p = SegPlan();
}

cudaError_t seg_plan_build(const CsrView& A, SegPlan* out, int capacity, bool force, cudaStream_t stream) {
    *out = SegPlan();
    if (A.rows <= 0 || A.nnz <= 0 || A.cols <= 0 || A.cols > static_cast<int>(kIdxMask)) return cudaSuccess;
    if (!force && !seg_worthwhile(A)) return cudaSuccess;
    const int device_cap = seg_table_capacity();
    if (device_cap < 4) return cudaSuccess;
    const bool whole_x = A.cols <= (capacity > 0 ? (capacity < device_cap ? capacity : device_cap) : device_cap);
    if (capacity <= 0) capacity = seg_default_capacity();
    if (capacity > device_cap) capacity = device_cap;

    SegPlan P;
    P.rows = A.rows; P.cols = A.cols; P.nnz = A.nnz;
    P.num_tiles = (A.nnz + kTile - 1) / kTile;
    const size_t padded = static_cast<size_t>(P.num_tiles) * kTile;
    if (padded > 0x7fffffffull) return cudaSuccess;  // int32 non-zero indices inside the kernel
    int* d_slot_of = nullptr;
    unsigned char* d_flags = nullptr;
    int* d_count = nullptr;
    void* d_temp = nullptr;
    auto fail = [&](cudaError_t e) {
        cudaGetLastError();
        cudaFree(d_slot_of); cudaFree(d_flags); cudaFree(d_count); cudaFree(d_temp);
        seg_plan_release(&P);
        return e;
    };
    cudaError_t e;
    if (whole_x) {
        P.whole_x = true;
        P.n_hot = A.cols;
        P.hot_nnz = A.nnz;
    } else {
        // a hub column is fetched once per CTA, so it must be referenced more often than there are CTAs
        const int t_min = force ? 2 : 2 * device_sm_count();
        if ((e = hot_select_columns(A, capacity, t_min, &d_slot_of, &P.hot_cols, &P.n_hot, &P.hot_nnz, stream)) != cudaSuccess)
            return fail(e);
        if (P.n_hot == 0) {  // no hub at all: every gather goes to global memory
            cudaFree(P.hot_cols);
            P.hot_cols = nullptr;
            cudaFree(d_slot_of);
            d_slot_of = nullptr;
            if ((e = cudaMalloc(&d_slot_of, sizeof(int) * static_cast<size_t>(A.cols))) != cudaSuccess) return fail(e);
            cudaMemsetAsync(d_slot_of, 0xff, sizeof(int) * static_cast<size_t>(A.cols), stream);  // all -1
        }
    }
    const size_t words = (static_cast<size_t>(A.rows) + 31) / 32;
    P.epilogue_blocks = static_cast<int>(plan_grid(A.rows));
    if ((e = cudaMalloc(&P.enc, sizeof(int) * padded)) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&P.rows_nz, sizeof(int) * static_cast<size_t>(A.rows))) != cudaSuccess) return fail(e);
    const int num_spans = P.num_tiles * kWarps;
    if ((e = cudaMalloc(&P.tile_head_base, sizeof(int) * (static_cast<size_t>(num_spans) + 1))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&P.nonempty, sizeof(uint32_t) * words)) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&P.tile_lead, sizeof(float) * static_cast<size_t>(P.num_tiles))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&P.tile_tail, sizeof(float) * static_cast<size_t>(P.num_tiles))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&P.partials, sizeof(double) * 3 * static_cast<size_t>(P.epilogue_blocks))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&d_flags, static_cast<size_t>(A.rows))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&d_count, sizeof(int))) != cudaSuccess) return fail(e);

    seg_encode_kernel<<<plan_grid(static_cast<long long>(padded)), kBlock, 0, stream>>>(
        A.nnz, static_cast<int>(padded), A.cols, A.col_indices, whole_x ? nullptr : d_slot_of, P.enc);
    seg_heads_kernel<<<plan_grid(A.rows), kBlock, 0, stream>>>(A.rows, A.row_ptrs, P.enc, d_flags, P.nonempty);
    count_launches(2);
    size_t temp_bytes = 0;
    thrust::counting_iterator<int> ids(0);
    if ((e = cub::DeviceSelect::Flagged(nullptr, temp_bytes, ids, d_flags, P.rows_nz, d_count, A.rows, stream)) != cudaSuccess)
        return fail(e);
    if ((e = cudaMalloc(&d_temp, temp_bytes ? temp_bytes : 16)) != cudaSuccess) return fail(e);
    if ((e = cub::DeviceSelect::Flagged(d_temp, temp_bytes, ids, d_flags, P.rows_nz, d_count, A.rows, stream)) != cudaSuccess)
        return fail(e);
    if ((e = cudaMemcpyAsync(&P.nonempty_rows, d_count, sizeof(int), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return fail(e);
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return fail(e);
    seg_span_heads_kernel<<<(num_spans + 1 + kBlock - 1) / kBlock, kBlock, 0, stream>>>(num_spans, P.nonempty_rows,
                                                                                       A.row_ptrs, P.rows_nz, P.tile_head_base);
    count_launches(1);
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return fail(e);
    if ((e = cudaGetLastError()) != cudaSuccess) return fail(e);
    cudaFree(d_slot_of); cudaFree(d_flags); cudaFree(d_count); cudaFree(d_temp);
    *out = P;
    return cudaSuccess;
}

cudaError_t launch_seg_spmv(const CsrView& A, const SegPlan& plan, const float* x, float* y, cudaStream_t stream) {
    if (A.rows <= 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(y, 0, sizeof(float) * static_cast<size_t>(A.rows), stream);  // rows without non-zeros
    if (e != cudaSuccess) return e;
    return run_seg(plan, A.values, x, y, stream);
}

cudaError_t launch_seg_pagerank(const CsrView& A, const SegPlan& plan, const PageRankStepArgs& args, cudaStream_t stream) {
    if (A.rows <= 0) return cudaMemsetAsync(args.out, 0, 3 * sizeof(double), stream);
    cudaError_t e = run_seg(plan, A.values, args.r_old, args.r_new + args.row_offset, stream);
    if (e != cudaSuccess) return e;
    seg_pagerank_epilogue_kernel<<<plan.epilogue_blocks, kBlock, 0, stream>>>(args, A.rows, plan.nonempty, plan.partials);
    count_launches(1);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return launch_reduce_partials(plan.partials, plan.epilogue_blocks, args.out, stream);
}

}  // namespace b200
}  // namespace spmv
