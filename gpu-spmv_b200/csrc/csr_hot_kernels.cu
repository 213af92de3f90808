// csr_hot_kernels.cu -- merge-path CSR SpMV for scale-free matrices: persistent
// CTAs that keep the x entries of the HUB COLUMNS in shared memory.
//
// Why.  On a power-law matrix the one-tile-per-CTA merge-path kernel
// (csr_merge_kernels.cu) is not limited by HBM but by the LSU data pipe of the L1TEX:
// a scattered 4-byte gather costs one wavefront per distinct 128-byte line and an SM
// retires one wavefront per clock (ncu on R-MAT 24: data pipe 77 % busy, DRAM 22 %, DRAM
// traffic = the compulsory bytes; profiles/r1_hub_kernel.md).  A scale-free matrix
// concentrates its non-zeros on few columns (R-MAT 24: the 24 K most referenced of
// 16.7 M columns carry 33 % of the non-zeros, the 48 K most referenced 44 %), so those
// x entries are copied ONCE per CTA into a shared-memory table; a table lookup costs a
// fraction of a wavefront (1-3 bank-conflict phases per 32 lanes).
//
// How.  A column plan (HotPlan), built once per matrix on the device:
//   1. per-column reference counts (atomics over col_indices),
//   2. the count threshold that admits at most `capacity` columns,
//   3. a slot per admitted column,
//   4. enc[j] = hub ? ~slot : col -- a private re-encoding of col_indices (the
//      caller's arrays are never modified).
// The kernel is the canonical two-level merge path (same coordinates, same
// carry fix-up, same row epilogues as csr_merge_kernels.cu, replacing reference
// src/spmv_kernels.cu:48-130,267) run by a persistent grid of one 1024-thread
// CTA per SM.  A CTA = 4 independent 256-thread workers (named barriers), each
// walking tiles w, w + stride, ...; the table is shared by the 4 workers.  A worker
// loads the next tile's values / enc span into the registers the current tile no longer
// needs, right before it starts reducing it, so the stream latency is off the critical
// path.  The table defaults to 24 576 entries (96 KB), NOT the 192 KB that would fit:
// shared memory is carved out of the L1's 256 KB and the L1's lines track the gather
// misses in flight (49 K entries: 46 % pipe utilisation, 1.86 ms against 1.04 ms).
// When the whole x fits the table (cols <= 49 152) no re-encoding is needed.
//
// Numerics: products and the per-thread serial order are those of the tile
// kernel; tiles are identical, so results are bit-identical to MERGE_PATH
// without the plan (tests/test_gpu_hot.py).
//
// Roofline: HBM, algorithmic bytes as for every CSR kernel (8*nnz + 4*(rows+1) +
// 4*cols + 4*rows, reference src/bandwidth.cpp:34-42); enc replaces col_indices
// in the stream, so the traffic is unchanged.  Measured: R-MAT 24 1.04 ms = 2.26 TB/s
// = 34.5 % of the measured HBM peak (tile kernel: 1.27 ms); the data pipe is 68 % busy.
#include "merge_rows.cuh"

#include <climits>
#include <cstdlib>
#include <cstring>

namespace spmv {
namespace b200 {
namespace {

constexpr int kWorkers = 4;
constexpr int kHotThreads = kWorkers * kT;  // 1024
// words per worker: product span (padded to 4), then row ends.  The tile is 256 * IPT merge items, IPT = 7 or 8
// chosen per matrix by merge_items_for() -- the SAME choice as the plain tile kernel's, so that a plan stays
// bit-identical to spmv_csr(MERGE_PATH) on every matrix.
constexpr int hot_buf_words(int ipt) { return kT * ipt + 8; }
constexpr int kWarps = kT / 32;             // warps per worker
constexpr int kCountBuckets = 65536;

__device__ __forceinline__ void worker_sync(int w) {
    asm volatile("bar.sync %0, %1;" :: "r"(w + 1), "n"(kT) : "memory");
}

// x entry of an encoded column: e < 0 -> slot ~e of the shared-memory table, else x[e].
// Predicated, not branched: a lane that reads the table issues no L1 wavefront.
__device__ __forceinline__ float gather_enc_hint(int e, uint32_t s_hot_addr, const float* __restrict__ x, uint64_t policy) {
    float r;
    const uint32_t sa = s_hot_addr + (static_cast<uint32_t>(~e) << 2);
    const unsigned long long ga = reinterpret_cast<unsigned long long>(x) +
                                  static_cast<unsigned long long>(static_cast<long long>(e) * 4);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.lt.s32 p, %1, 0;\n"
        "@p ld.shared.f32 %0, [%2];\n"
        "@!p ld.global.nc.L2::cache_hint.f32 %0, [%3], %4;\n"
        "}\n"
        : "=f"(r)
        : "r"(e), "r"(sa), "l"(ga), "l"(policy));
    return r;
}

__device__ __forceinline__ float gather_enc(int e, uint32_t s_hot_addr, const float* __restrict__ x) {
    float r;
    const uint32_t sa = s_hot_addr + (static_cast<uint32_t>(~e) << 2);
    const unsigned long long ga = reinterpret_cast<unsigned long long>(x) +
                                  static_cast<unsigned long long>(static_cast<long long>(e) * 4);
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

// One tile's share of the matrix stream held by a thread: kIPT single non-zeros, lane-consecutive
// (a warp-wide gather covers 32 ADJACENT non-zeros; 32-bit loads, so no alignment requirement).
template <int IPT>
struct StreamRegs {
    float v[IPT];
    int c[IPT];
};

// l2_mode bit 0: the stream is loaded with L2::evict_first (read once; must not displace x in L2)
template <int kIPT>
__device__ __forceinline__ void load_stream(StreamRegs<kIPT>& s, int nz_s, int nz_e, int wt,
                                            const float* __restrict__ values, const int* __restrict__ enc,
                                            unsigned l2_mode, uint64_t pol_first) {
    if (l2_mode & 1u) {
#pragma unroll
        for (int u = 0; u < kIPT; ++u) {
            const int j = nz_s + wt + u * kT;
            if (j < nz_e) {
                s.v[u] = dev::ld_stream_f_hint(values + j, pol_first);
                s.c[u] = dev::ld_stream_i_hint(enc + j, pol_first);
            }
        }
        return;
    }
#pragma unroll
    for (int u = 0; u < kIPT; ++u) {
        const int j = nz_s + wt + u * kT;
        if (j < nz_e) {
            s.v[u] = dev::ld_stream_f(values + j);
            s.c[u] = dev::ld_stream_i(enc + j);
        }
    }
}

// l2_mode bit 1: cold gathers carry L2::evict_last (x is what should stay in L2)
template <bool ALL_HOT>
__device__ __forceinline__ float gather_one(int e, const float* s_hot, uint32_t s_hot_addr,
                                            const float* __restrict__ x, unsigned l2_mode, uint64_t pol_last) {
    if (ALL_HOT) return s_hot[e];
    if (l2_mode & 2u) return gather_enc_hint(e, s_hot_addr, x, pol_last);
    return gather_enc(e, s_hot_addr, x);
}

__device__ __forceinline__ void worker_store_sums(const RankSums& s, double* __restrict__ partials, int slot,
                                                  double (*scratch)[3], int w, int wt) {
    double a = dev::warp_sum(s.l2), b = dev::warp_sum(s.l1), c = dev::warp_sum(s.dangling);
    const int warp = wt >> 5;
    if ((wt & 31) == 0) { scratch[warp][0] = a; scratch[warp][1] = b; scratch[warp][2] = c; }
    worker_sync(w);
    if (wt < 3) {
        double t = 0.0;
        for (int k = 0; k < kWarps; ++k) t += scratch[k][wt];
        partials[static_cast<size_t>(slot) * 3 + wt] = t;
    }
}
__device__ __forceinline__ void worker_store_sums(const NoSums&, double*, int, double (*)[3], int, int) {}

// Shared memory: [hot table: hot_slots floats][kWorkers x kBuf words][kWorkers x kWarps x 3 doubles]
//                [kWorkers x kWarps floats][kWorkers x kWarps ints]
constexpr size_t hot_fixed_smem(int ipt) {
    return static_cast<size_t>(kWorkers) * hot_buf_words(ipt) * 4 + kWorkers * kWarps * (3 * 8 + 4 + 4);
}
constexpr size_t kHotFixedSmem = hot_fixed_smem(8);  // the larger geometry: what the table capacity is sized against

// One CTA per SM (64 registers per thread); the next tile's stream is loaded into registers while
// the current tile is reduced.  (Two CTAs of 32 registers per SM spill and measured 1.7x slower.)
// Measured dead ends (R-MAT 24, profiles/r1_hub_kernel.md): cold gathers through the texture pipe
// (TLD) 5-8 % slower than LDG; L1::no_allocate gathers 3-20 % slower; two 32-register CTAs per SM
// spill and run 1.7x slower; 128-bit stream loads (4 non-zeros per lane) 1 % slower.  Round 2: a deeper software
// pipeline (x gathers + values of tile k+1 and columns of tile k+2 issued before tile k is reduced, same
// register count, bit-identical) made the product 12 % SLOWER (1.168 against 1.039 ms) and left the PageRank
// step unchanged: more gathers in flight only lengthen the queue in front of the L1 miss path, which is
// what the kernel is bound by (scripts/microbench/gather_bench.cu: L2-resident gathers retire at 1 per clock
// and SM, L1-resident ones at 2.3, shared-memory ones at 4.4).
template <class Row, bool ALL_HOT, int IPT>
__global__ void __launch_bounds__(kHotThreads, 1)
merge_hot_kernel(int rows, int nnz, const int* __restrict__ row_ptrs, const int* __restrict__ enc,
                 const float* __restrict__ values, const float* __restrict__ x,
                 const int* __restrict__ hot_cols, int n_hot, const int2* __restrict__ coords, int num_tiles,
                 int* __restrict__ carry_row, float* __restrict__ carry_val, Row row_op,
                 double* __restrict__ partials, unsigned l2_mode) {
    constexpr int kIPT = IPT;  // shadow the file-level geometry: this kernel's tile is kT * IPT items
    constexpr int kBuf = kT * IPT + 8;  // == hot_buf_words(IPT)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint64_t pol_first = dev::l2_policy_evict_first();
    const uint64_t pol_last = dev::l2_policy_evict_last();
    const int hot_slots = (n_hot + 3) & ~3;
    float* s_hot = reinterpret_cast<float*>(smem_raw);
    const int tid = threadIdx.x;
    const int w = tid / kT;   // worker
    const int wt = tid % kT;  // thread inside the worker
    float* s_prod = s_hot + hot_slots + w * kBuf;
    unsigned char* after = reinterpret_cast<unsigned char*>(s_hot + hot_slots + kWorkers * kBuf);
    double (*s_sums)[3] = reinterpret_cast<double (*)[3]>(after) + w * kWarps;
    float* s_warp_val = reinterpret_cast<float*>(after + kWorkers * kWarps * 24) + w * kWarps;
    int* s_warp_flag = reinterpret_cast<int*>(after + kWorkers * kWarps * 28) + w * kWarps;

    // ---- the table: x of the hub columns (or all of x), once per CTA ----------------
    for (int i = tid; i < hot_slots; i += kHotThreads)
        s_hot[i] = i < n_hot ? dev::ld_x(x + (ALL_HOT ? i : __ldg(hot_cols + i))) : 0.0f;
    __syncthreads();
    const uint32_t s_hot_addr = dev::smem_u32(s_hot);

    const int stride = gridDim.x * kWorkers;
    int tile = w * gridDim.x + blockIdx.x;

    typename Row::Sums sums;
    sums.clear();
    const float row_ctx = row_op.prepare();

    int2 c0 = make_int2(0, 0), c1 = c0;
    StreamRegs<IPT> cur;
    if (tile < num_tiles) {
        c0 = __ldg(coords + tile);
        c1 = __ldg(coords + tile + 1);
        load_stream(cur, c0.y, c1.y, wt, values, enc, l2_mode, pol_first);
    }

    while (tile < num_tiles) {
        const int next = tile + stride;
        const int row_s = c0.x, nz_s = c0.y, nz_e = c1.y;
        const int tile_rows = c1.x - c0.x;
        const int tile_nz = nz_e - nz_s;
        const int tile_items = tile_rows + tile_nz;
        const int base = nz_s;                         // s_prod slot of non-zero j is j - base
        const int ends_at = ((nz_e - base) + 3) & ~3;  // row ends follow the product span
        int* s_end = reinterpret_cast<int*>(s_prod) + ends_at;
        int2 n0 = c0, n1 = c1;
        if (next < num_tiles) {  // consumed after the gathers have been issued
            n0 = __ldg(coords + next);
            n1 = __ldg(coords + next + 1);
        }

        // ---- x gathers of this thread's share of the span (all issued before the first use) ----
        float xv[kIPT];
#pragma unroll
        for (int u = 0; u < kIPT; ++u)
            if (nz_s + wt + u * kT < nz_e) xv[u] = gather_one<ALL_HOT>(cur.c[u], s_hot, s_hot_addr, x, l2_mode, pol_last);
        // ---- row ends of the tile (tile_rows + 1 entries; the last bounds the open row) ----
        for (int i0 = wt; i0 <= tile_rows; i0 += 4 * kT) {
            int e[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = i0 + k * kT;
                if (i <= tile_rows) e[k] = (row_s + i < rows) ? dev::ld_stream_i(row_ptrs + row_s + 1 + i) : INT_MAX;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = i0 + k * kT;
                if (i <= tile_rows) s_end[i] = e[k];
            }
        }
        // does the tile's first row own non-zeros in earlier tiles?
        const int first_row_start = (row_s < rows) ? __ldg(row_ptrs + row_s) : nz_e;
        // ---- products of [nz_s, nz_e) at slot (j - base) -----------------------------------
#pragma unroll
        for (int u = 0; u < kIPT; ++u) {
            const int j = nz_s + wt + u * kT;
            if (j < nz_e) s_prod[j - base] = cur.v[u] * xv[u];
        }
        // ---- next tile's stream: in flight while this tile is reduced ----------------------
        if (next < num_tiles) load_stream(cur, n0.y, n1.y, wt, values, enc, l2_mode, pol_first);
        const bool first_row_split = (row_s < rows) && (nz_s > first_row_start);
        worker_sync(w);

        // ---- per-thread diagonal inside the tile (search in shared memory) -----------------
        const int diag = min(wt * kIPT, tile_items);
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
        // start of the row left open at the tile end (read before the buffers may be reused)
        int open_start = 0;
        if (wt == kT - 1) open_start = tile_rows > 0 ? s_end[tile_rows - 1] : first_row_start;

        // ---- segmented scan of (emitted, running) over the worker ---------------------------
        const int lane = wt & 31, warp = wt >> 5;
        float v = running;
        int f, ex_f;
        float ex_v;
        warp_segmented_scan(v, emitted, lane, f, ex_v, ex_f);
        if (lane == 31) { s_warp_val[warp] = v; s_warp_flag[warp] = f; }
        worker_sync(w);  // from here on nobody reads s_prod / s_end of this tile
        float pre_v = 0.0f;
        int pre_f = 0;
        for (int k = 0; k < warp; ++k) {
            const float wv = s_warp_val[k];
            const int wf = s_warp_flag[k];
            pre_v = wf ? wv : pre_v + wv;
            pre_f |= wf;
        }
        const float carry_in = ex_f ? ex_v : pre_v + ex_v;

        if (emitted) {
            const float total = carry_in + first_sum;
            if (first_row == 0 && first_row_split) row_op.park(row_s, total);  // the fix-up finishes it
            else row_op.tile_finish(row_s + first_row, total, sums, row_ctx);
        }
        if (wt == kT - 1) {  // tile carry-out: the row still open at the tile end
            const float open_sum = f ? v : pre_v + v;
            const int row_e = c1.x;
            const bool has_open = (row_e < rows) && (nz_e > max(open_start, nz_s));
            carry_row[tile] = has_open ? row_e : -1;
            carry_val[tile] = has_open ? open_sum : 0.0f;
        }
        if (Row::kReduces) {
            worker_sync(w);  // every raw row sum of this tile is visible to the worker
            row_op.tile_epilogue(row_s + (first_row_split ? 1 : 0), c1.x, wt, sums, row_ctx);
        }
        // The next tile's buffers are written before its first barrier; every thread has left the
        // reads of this tile behind at the barrier above, and s_warp_val / s_warp_flag are only
        // rewritten after the next tile's first barrier, which the slowest folder must reach first.
        tile = next;
        c0 = n0;
        c1 = n1;
    }
    if (Row::kReduces) worker_store_sums(sums, partials, blockIdx.x * kWorkers + w, s_sums, w, wt);
}

// ------------------------------------------------------------------ plan kernels ----

constexpr int kPlanBlock = 256;
inline unsigned plan_grid(long long n) {
    long long b = (n + kPlanBlock - 1) / kPlanBlock;
    if (b < 1) b = 1;
    return static_cast<unsigned>(b < 148 * 16 ? b : 148 * 16);
}

__global__ void hot_count_kernel(int nnz, int cols, const int* __restrict__ col_indices, int* __restrict__ counts) {
    for (long long j = blockIdx.x * static_cast<long long>(kPlanBlock) + threadIdx.x; j < nnz;
         j += static_cast<long long>(gridDim.x) * kPlanBlock) {
        const int c = dev::ld_stream_i(col_indices + j);
        if (c >= 0 && c < cols) atomicAdd(counts + c, 1);
    }
}

// histogram of the reference counts that could qualify (count >= t_min), clamped to the last bucket
__global__ void hot_hist_kernel(int cols, const int* __restrict__ counts, int t_min, unsigned* __restrict__ hist) {
    for (long long c = blockIdx.x * static_cast<long long>(kPlanBlock) + threadIdx.x; c < cols;
         c += static_cast<long long>(gridDim.x) * kPlanBlock) {
        const int n = counts[c];
        if (n >= t_min) atomicAdd(hist + min(n, kCountBuckets - 1), 1u);
    }
}

// smallest threshold T >= t_min with #(count >= T) <= capacity (one CTA of 1024 threads)
__global__ void __launch_bounds__(1024)
hot_threshold_kernel(const unsigned* __restrict__ hist, int capacity, int t_min, int* __restrict__ out_t) {
    __shared__ unsigned s_chunk[1024];
    __shared__ unsigned s_above[1024];
    __shared__ int s_t;
    constexpr int per = kCountBuckets / 1024;
    const int t = threadIdx.x;
    unsigned sum = 0;
    for (int b = 0; b < per; ++b) sum += hist[t * per + b];
    s_chunk[t] = sum;
    if (t == 0) s_t = t_min;
    __syncthreads();
    if (t == 0) {
        unsigned acc = 0;
        for (int u = 1023; u >= 0; --u) {
            s_above[u] = acc;  // entries in the chunks above u
            acc += s_chunk[u];
        }
    }
    __syncthreads();
    unsigned running = s_above[t];
    for (int b = per - 1; b >= 0; --b) {
        running += hist[t * per + b];
        if (running > static_cast<unsigned>(capacity)) {  // bucket t*per+b does not fit any more
            atomicMax(&s_t, t * per + b + 1);
            break;
        }
    }
    __syncthreads();
    if (t == 0) *out_t = s_t;
}

// counts[c] becomes the slot of column c (or -1); slots past `capacity` stay cold, so the plan is
// valid whatever the threshold.  stats[0] = admitted columns (unclamped), stats64 = their non-zeros.
__global__ void hot_assign_kernel(int cols, int* __restrict__ counts, const int* __restrict__ d_t, int capacity,
                                  int* __restrict__ hot_cols, int* __restrict__ n_admitted,
                                  unsigned long long* __restrict__ hot_nnz) {
    const int threshold = *d_t;
    for (long long c = blockIdx.x * static_cast<long long>(kPlanBlock) + threadIdx.x; c < cols;
         c += static_cast<long long>(gridDim.x) * kPlanBlock) {
        const int n = counts[c];
        int slot = -1;
        if (n >= threshold) {
            slot = atomicAdd(n_admitted, 1);
            if (slot < capacity) {
                hot_cols[slot] = static_cast<int>(c);
                atomicAdd(hot_nnz, static_cast<unsigned long long>(n));
            } else {
                slot = -1;
            }
        }
        counts[c] = slot;
    }
}

__global__ void hot_encode_kernel(int nnz, int cols, const int* __restrict__ col_indices,
                                  const int* __restrict__ slot_of, int* __restrict__ enc) {
    for (long long j = blockIdx.x * static_cast<long long>(kPlanBlock) + threadIdx.x; j < nnz;
         j += static_cast<long long>(gridDim.x) * kPlanBlock) {
        const int c = dev::ld_stream_i(col_indices + j);
        int e = c;
        if (c >= 0 && c < cols) {
            const int s = __ldg(slot_of + c);
            if (s >= 0) e = ~s;
        }
        enc[j] = e;
    }
}

int device_sms() {
    int sms = 148, dev_id = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
    return sms;
}

template <class Row, bool ALL_HOT, int IPT>
cudaError_t run_hot_variant(const CsrView& A, const HotPlan& hot, const float* x, const MergePlan& plan,
                            const Row& row_op, cudaStream_t stream, int* grid_out) {
    const int sms = device_sms();
    const int n_hot = ALL_HOT ? A.cols : hot.n_hot;
    const size_t smem = static_cast<size_t>((n_hot + 3) & ~3) * 4 + hot_fixed_smem(IPT);
    auto kernel = merge_hot_kernel<Row, ALL_HOT, IPT>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    // L2 priorities (bit 0: stream evict_first, bit 1: x gathers evict_last).  Default: on when x does not
    // fit L2 comfortably (> 64 MB), where the 8 B/nnz stream would otherwise push x out; SPMV_B200_HOT_L2 forces.
    static const int env_l2 = env_int("SPMV_B200_HOT_L2", -1);
    const int l2_mode = env_l2 >= 0 ? env_l2 : 0;
    int grid = sms;  // persistent: one CTA per SM
    if (grid > plan.num_tiles / kWorkers) grid = plan.num_tiles / kWorkers;  // per-worker sums fit plan.partials
    if (grid < 1) grid = 1;
    if (grid_out) *grid_out = grid;
    kernel<<<grid, kHotThreads, smem, stream>>>(A.rows, A.nnz, A.row_ptrs, ALL_HOT ? A.col_indices : hot.enc, A.values, x,
                                                ALL_HOT ? nullptr : hot.hot_cols, n_hot, plan.coords, plan.num_tiles,
                                                plan.carry_row, plan.carry_val, row_op, plan.partials,
                                                static_cast<unsigned>(l2_mode));
    count_launches(1);
    return cudaGetLastError();
}

template <class Row>
cudaError_t run_hot(const CsrView& A, const HotPlan& hot, const float* x, const MergePlan& plan, const Row& row_op,
                    cudaStream_t stream, int* grid_out) {
    // 8-item tiles exist for the plain product only (the PageRank plans are always cut at 7 items)
    if (!Row::kReduces && plan.ipt == 8) {
        if (hot.all_hot) return run_hot_variant<Row, true, (Row::kReduces ? kIPT : 8)>(A, hot, x, plan, row_op, stream, grid_out);
        return run_hot_variant<Row, false, (Row::kReduces ? kIPT : 8)>(A, hot, x, plan, row_op, stream, grid_out);
    }
    if (plan.ipt != kIPT) return cudaErrorInvalidValue;
    if (hot.all_hot) return run_hot_variant<Row, true, kIPT>(A, hot, x, plan, row_op, stream, grid_out);
    return run_hot_variant<Row, false, kIPT>(A, hot, x, plan, row_op, stream, grid_out);
}

}  // namespace

// ------------------------------------------------------------------------ host side ----

int device_sm_count() { return device_sms(); }

int hot_capacity() {
    int dev_id = 0, optin = 0;
    cudaGetDevice(&dev_id);
    if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev_id) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    const long long room = static_cast<long long>(optin) - static_cast<long long>(kHotFixedSmem) - 64;
    return room > 0 ? static_cast<int>(room / 4) & ~1023 : 0;
}

// Table size used when the caller does not ask for one.  NOT the maximum: shared memory is carved
// out of the same 256 KB as the L1, and the L1's lines are what tracks the outstanding gather
// misses -- with the 192 KB table ncu shows the data pipe at 48 % and the kernel 50 % slower than
// with 64-128 KB (profiles/r1_hub_kernel.md).
int hot_default_capacity() {
    static const int env_cap = env_int("SPMV_B200_HOT_CAP", 0);
    const int cap = hot_capacity();
    const int want = env_cap > 0 ? (env_cap & ~3) : 24576;
    return want < cap ? want : cap;
}

bool hot_worthwhile(const CsrView& A) {
    // the persistent grid needs a few tiles per worker; below that the tile kernel wins
    return merge_num_tiles(A.rows, A.nnz) >= kWorkers * device_sms() * 4;
}

void hot_plan_release(HotPlan* p) {
    if (!p) return;
    if (p->enc) cudaFree(p->enc);
    if (p->hot_cols) cudaFree(p->hot_cols);
    *p = HotPlan();
}

// The `capacity` most referenced columns (reference count >= t_min): *d_slot_of (device int[cols],
// caller frees) maps a column to its table slot or -1, *d_hot_cols (device int[capacity], caller
// frees) is the inverse.  Synchronises `stream`.
cudaError_t hot_select_columns(const CsrView& A, int capacity, int t_min, int** d_slot_of, int** d_hot_cols_out,
                               int* n_hot_out, long long* hot_nnz_out, cudaStream_t stream) {
    int* d_counts = nullptr;
    unsigned* d_hist = nullptr;
    int* d_small = nullptr;  // [0] threshold, [1] admitted, [2..3] hot nnz (64-bit)
    int* d_hot_cols = nullptr;
    auto fail = [&](cudaError_t e) {
        cudaGetLastError();
        cudaFree(d_counts); cudaFree(d_hist); cudaFree(d_small); cudaFree(d_hot_cols);
        return e;
    };
    cudaError_t e;
    if ((e = cudaMalloc(&d_counts, sizeof(int) * static_cast<size_t>(A.cols))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&d_hist, sizeof(unsigned) * kCountBuckets)) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&d_small, 4 * sizeof(int))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&d_hot_cols, sizeof(int) * static_cast<size_t>(capacity))) != cudaSuccess) return fail(e);
    cudaMemsetAsync(d_counts, 0, sizeof(int) * static_cast<size_t>(A.cols), stream);
    cudaMemsetAsync(d_hist, 0, sizeof(unsigned) * kCountBuckets, stream);
    cudaMemsetAsync(d_small, 0, 4 * sizeof(int), stream);
    hot_count_kernel<<<plan_grid(A.nnz), kPlanBlock, 0, stream>>>(A.nnz, A.cols, A.col_indices, d_counts);
    hot_hist_kernel<<<plan_grid(A.cols), kPlanBlock, 0, stream>>>(A.cols, d_counts, t_min, d_hist);
    hot_threshold_kernel<<<1, 1024, 0, stream>>>(d_hist, capacity, t_min, d_small);
    hot_assign_kernel<<<plan_grid(A.cols), kPlanBlock, 0, stream>>>(A.cols, d_counts, d_small, capacity, d_hot_cols,
                                                                   d_small + 1,
                                                                   reinterpret_cast<unsigned long long*>(d_small + 2));
    count_launches(4);
    int h_small[4] = {0, 0, 0, 0};
    if ((e = cudaMemcpyAsync(h_small, d_small, sizeof(h_small), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return fail(e);
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return fail(e);
    unsigned long long hot_nnz = 0;
    memcpy(&hot_nnz, h_small + 2, sizeof(hot_nnz));
    cudaFree(d_hist);
    cudaFree(d_small);
    *d_slot_of = d_counts;
    *d_hot_cols_out = d_hot_cols;
    *n_hot_out = h_small[1] < capacity ? h_small[1] : capacity;
    *hot_nnz_out = static_cast<long long>(hot_nnz);
    return cudaSuccess;
}

cudaError_t hot_plan_build(const CsrView& A, HotPlan* out, int capacity, bool force, cudaStream_t stream,
                           int min_share) {
    *out = HotPlan();
    out->nnz = A.nnz;
    out->cols = A.cols;
    const int device_cap = hot_capacity();
    const bool whole_x = A.cols <= (capacity > 0 ? (capacity < device_cap ? capacity : device_cap) : device_cap);
    if (capacity <= 0) capacity = hot_default_capacity();
    if (capacity > device_cap) capacity = device_cap;
    if (A.rows <= 0 || A.nnz <= 0 || A.cols <= 0 || capacity < 4) return cudaSuccess;
    if (!force && !hot_worthwhile(A)) return cudaSuccess;
    if (whole_x) {  // x itself is the table: no global gather is left, so the size costs nothing
        out->all_hot = true;
        out->n_hot = A.cols;
        out->hot_nnz = A.nnz;
        return cudaSuccess;
    }
    // A hub column is fetched once per CTA, so it must be referenced more often than there are CTAs
    const int t_min = force ? 2 : 2 * device_sms();
    int* d_slot_of = nullptr;
    int* d_hot_cols = nullptr;
    int n_hot = 0;
    long long hot_nnz = 0;
    cudaError_t e = hot_select_columns(A, capacity, t_min, &d_slot_of, &d_hot_cols, &n_hot, &hot_nnz, stream);
    if (e != cudaSuccess) return e;
    // worth it when the table takes a real share of the gathers off the L1
    const bool useful = n_hot > 0 && (force || hot_nnz * min_share >= static_cast<long long>(A.nnz));
    int* d_enc = nullptr;
    if (useful && (e = cudaMalloc(&d_enc, sizeof(int) * static_cast<size_t>(A.nnz))) == cudaSuccess) {
        hot_encode_kernel<<<plan_grid(A.nnz), kPlanBlock, 0, stream>>>(A.nnz, A.cols, A.col_indices, d_slot_of, d_enc);
        count_launches(1);
        e = cudaStreamSynchronize(stream);
    }
    cudaFree(d_slot_of);
    if (!useful || e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d_enc);
        cudaFree(d_hot_cols);
        return useful ? e : cudaSuccess;
    }
    out->enc = d_enc;
    out->hot_cols = d_hot_cols;
    out->n_hot = n_hot;
    out->hot_nnz = hot_nnz;
    return cudaSuccess;
}

cudaError_t launch_hot_spmv(const CsrView& A, const HotPlan& hot, const float* x, float* y, const MergePlan& plan,
                            cudaStream_t stream) {
    if (A.rows <= 0 || plan.num_tiles <= 0) return cudaSuccess;
    PlainRow op{y};
    cudaError_t e = run_hot(A, hot, x, plan, op, stream, nullptr);
    if (e != cudaSuccess) return e;
    return launch_merge_fixup(plan, y, stream);
}

cudaError_t launch_hot_pagerank(const CsrView& A, const HotPlan& hot, const MergePlan& plan,
                                const PageRankStepArgs& args, cudaStream_t stream) {
    if (A.rows <= 0 || plan.num_tiles <= 0) return cudaMemsetAsync(args.out, 0, 3 * sizeof(double), stream);
    PageRankRowT<true> op{args};
    int grid = 0;
    cudaError_t e = run_hot(A, hot, args.r_old, plan, op, stream, &grid);
    if (e != cudaSuccess) return e;
    return launch_merge_fixup_pagerank(plan, args, grid * kWorkers, stream);
}

}  // namespace b200
}  // namespace spmv
