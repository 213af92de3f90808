// csr_stream_kernels.cu -- row-owner CSR SpMV kernels for sm_100a
// (SCALAR_CSR and VECTOR_CSR of the reference API).
//
// Replaces spmv_csr_scalar_kernel / spmv_csr_vector_kernel (reference
// src/spmv_kernels.cu:168-188, :133-165).  The reference lets every row owner
// fetch its own non-zeros, so lanes stride by the row length (scalar) or most
// lanes idle on short rows (vector, 5-nnz rows use 5 of 32 lanes).
//
// csr_stream_kernel<LPR> separates the two jobs:
//   1. STAGE   a CTA owns a window of consecutive rows.  It stages the
//              window's row_ptrs in shared memory with one 1-D TMA bulk copy
//              (cp.async.bulk + mbarrier), then streams the window's
//              contiguous non-zero range with fully coalesced 128-bit loads of
//              values and col_indices (row boundaries are irrelevant here),
//              gathers x and parks the PRODUCTS in shared memory.
//   2. REDUCE  each row is owned by LPR lanes that sum the row's products out
//              of shared memory.
//      LPR == 1 (SCALAR_CSR): one thread, sequential order, separately rounded
//              multiply and add -> bit-identical to spmv_cpu_csr
//              (reference src/spmv_cpu.cpp:6-16).
//      LPR in {2,4,8,16} (VECTOR_CSR): lanes stride the row, shuffle tree.
//
// csr_warp_row_kernel is VECTOR_CSR for long rows (average >= 64): one warp per
// row, 128-bit loads on the 16-byte aligned interior of the row, shuffle tree.
//
// Roofline: HBM.  Algorithmic bytes per launch = 8*nnz + 4*(rows+1) + 4*cols +
// 4*rows (reference src/bandwidth.cpp:34-42).
#include "device_utils.cuh"
#include "internal.hpp"

#include <algorithm>
#include <mutex>
#include <unordered_map>

namespace spmv {
namespace b200 {
namespace {

constexpr int kThreads = 256;
constexpr int kProductCap = 5632;  // products parked per pass (22 KB)

// CTA geometry for LPR lanes per row: `groups` row owners, each holding at most
// `max_rows_per_group` running sums in registers.
template <int LPR>
struct StreamGeom {
    static constexpr int groups = kThreads / LPR;
    static constexpr int max_rows_per_group = (1024 / groups) < 8 ? (1024 / groups) : 8;
    static constexpr int max_window_rows = groups * max_rows_per_group;  // <= 1024
};

// shared-memory layout: [mbarrier 16 B][row window (R + 4) ints][products kProductCap floats]
__host__ __device__ constexpr size_t stream_smem_bytes(int window_rows) {
    return 16 + static_cast<size_t>(window_rows + 4) * sizeof(int) + kProductCap * sizeof(float);
}

template <int LPR>
__global__ void __launch_bounds__(kThreads)
csr_stream_kernel(int rows, int nnz, const int* __restrict__ row_ptrs,
                  const int* __restrict__ col_indices, const float* __restrict__ values,
                  const float* __restrict__ x, float* __restrict__ y, int window_rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    int* s_rp = reinterpret_cast<int*>(smem_raw + 16);
    float* s_prod = reinterpret_cast<float*>(smem_raw + 16 + static_cast<size_t>(window_rows + 4) * sizeof(int));

    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * window_rows;
    const int nr = min(window_rows, rows - r0);  // rows in this window (>= 1)

    // ---- stage row_ptrs[r0 .. r0 + nr] -------------------------------------
    // Full windows go through one TMA bulk copy of (window_rows + 4) ints (the
    // copy size must be a multiple of 16 bytes); ragged / unaligned windows
    // fall back to plain loads.
    const int* gp = row_ptrs + r0;
    const bool bulk = (nr == window_rows) && (r0 + window_rows + 4 <= rows + 1) && dev::aligned16(gp);
    if (bulk) {
        if (tid == 0) {
            dev::mbar_init(bar, 1);
            dev::mbar_fence_init();
        }
        __syncthreads();
        if (tid == 0) {
            const uint32_t bytes = static_cast<uint32_t>(window_rows + 4) * sizeof(int);
            dev::mbar_arrive_expect_tx(bar, bytes);
            dev::tma_bulk_g2s(s_rp, gp, bytes, bar);
        }
        dev::mbar_wait(bar, 0);
    } else {
        for (int i = tid; i <= nr; i += kThreads) s_rp[i] = row_ptrs[r0 + i];
        __syncthreads();
    }

    const int n0 = s_rp[0];
    const int n1 = s_rp[nr];

    constexpr int kGroups = StreamGeom<LPR>::groups;  // row owners per CTA
    constexpr int kMaxRowsPerGroup = StreamGeom<LPR>::max_rows_per_group;
    const int group = tid / LPR;
    const int lane = tid % LPR;
    float acc[kMaxRowsPerGroup];
#pragma unroll
    for (int i = 0; i < kMaxRowsPerGroup; ++i) acc[i] = 0.0f;

    // ---- passes over the window's non-zero range ----------------------------
    // `base` is 4-aligned so that 128-bit loads of values/col_indices are
    // aligned (when the arrays themselves are 16-byte aligned; any device
    // pointer is legal in the public struct, so that is checked here); slot
    // (j - base) of s_prod holds the product of non-zero j.
    const bool vec_ok = dev::aligned16(values) && dev::aligned16(col_indices);
    for (int base = n0 & ~3; base < n1; base += kProductCap) {
        const int hi = min(base + kProductCap, n1);  // exclusive end of this pass
        const int lo = max(base, n0);
        if (base != (n0 & ~3)) __syncthreads();      // previous pass fully reduced

        for (int j = base + 4 * tid; j < hi; j += 4 * kThreads) {
            float p0, p1, p2, p3;
            if (vec_ok && j >= lo && j + 4 <= hi) {
                const float4 v = dev::ld_stream_f4(values + j);
                const int4 c = dev::ld_stream_i4(col_indices + j);
                p0 = __fmul_rn(v.x, dev::ld_x(x + c.x));
                p1 = __fmul_rn(v.y, dev::ld_x(x + c.y));
                p2 = __fmul_rn(v.z, dev::ld_x(x + c.z));
                p3 = __fmul_rn(v.w, dev::ld_x(x + c.w));
            } else {  // ragged head / tail of the range
                p0 = (j + 0 >= lo && j + 0 < hi) ? __fmul_rn(values[j + 0], dev::ld_x(x + col_indices[j + 0])) : 0.0f;
                p1 = (j + 1 >= lo && j + 1 < hi) ? __fmul_rn(values[j + 1], dev::ld_x(x + col_indices[j + 1])) : 0.0f;
                p2 = (j + 2 >= lo && j + 2 < hi) ? __fmul_rn(values[j + 2], dev::ld_x(x + col_indices[j + 2])) : 0.0f;
                p3 = (j + 3 >= lo && j + 3 < hi) ? __fmul_rn(values[j + 3], dev::ld_x(x + col_indices[j + 3])) : 0.0f;
            }
            *reinterpret_cast<float4*>(s_prod + (j - base)) = make_float4(p0, p1, p2, p3);
        }
        __syncthreads();

        // ---- reduce: row owners pick up their rows' products -----------------
#pragma unroll
        for (int i = 0; i < kMaxRowsPerGroup; ++i) {
            const int r = group + i * kGroups;
            if (r < nr) {
                const int a = max(s_rp[r], lo);
                const int b = min(s_rp[r + 1], hi);
                float s = acc[i];
                for (int j = a + lane; j < b; j += LPR) s = __fadd_rn(s, s_prod[j - base]);
                acc[i] = s;
            }
        }
    }

    // ---- finish: combine lanes, write y ---------------------------------------
#pragma unroll
    for (int i = 0; i < kMaxRowsPerGroup; ++i) {
        float s = acc[i];
#pragma unroll
        for (int d = LPR / 2; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d, LPR);
        const int r = group + i * kGroups;
        if (lane == 0 && r < nr) y[r0 + r] = s;
    }
}

// One warp per row; rows are expected to be long (>= 64 non-zeros on average).
__global__ void __launch_bounds__(kThreads)
csr_warp_row_kernel(int rows, const int* __restrict__ row_ptrs, const int* __restrict__ col_indices,
                    const float* __restrict__ values, const float* __restrict__ x,
                    float* __restrict__ y) {
    const int warp = (blockIdx.x * kThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= rows) return;
    const int a = row_ptrs[warp];
    const int b = row_ptrs[warp + 1];
    const bool vec_ok = dev::aligned16(values) && dev::aligned16(col_indices);
    float s = 0.0f;
    // 4-element groups starting at the aligned address at or below `a`
    for (int j = (a & ~3) + 4 * lane; j < b; j += 128) {
        if (vec_ok && j >= a && j + 4 <= b) {
            const float4 v = dev::ld_stream_f4(values + j);
            const int4 c = dev::ld_stream_i4(col_indices + j);
            s = fmaf(v.x, dev::ld_x(x + c.x), s);
            s = fmaf(v.y, dev::ld_x(x + c.y), s);
            s = fmaf(v.z, dev::ld_x(x + c.z), s);
            s = fmaf(v.w, dev::ld_x(x + c.w), s);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (j + e >= a && j + e < b) s = fmaf(values[j + e], dev::ld_x(x + col_indices[j + e]), s);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
    if (lane == 0) y[warp] = s;
}

__global__ void zero_rows_kernel(int rows, float* __restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rows) y[i] = 0.0f;
}

// Window size: as many rows as keep the expected non-zero count of a window
// inside one product pass, limited to what the row owners can hold in
// registers, a multiple of the group count.
template <int LPR>
int pick_window_rows(int rows, int nnz) {
    constexpr int groups = StreamGeom<LPR>::groups;
    constexpr int max_mult = StreamGeom<LPR>::max_rows_per_group;
    const double avg = rows > 0 ? static_cast<double>(nnz) / rows : 0.0;
    int mult = max_mult;
    while (mult > 1 && avg * groups * mult > kProductCap - 8) mult >>= 1;
    return groups * mult;
}

template <int LPR>
cudaError_t launch_stream_lpr(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    const int window = pick_window_rows<LPR>(A.rows, A.nnz);
    const size_t smem = stream_smem_bytes(window);
    cudaError_t e = cudaFuncSetAttribute(csr_stream_kernel<LPR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(stream_smem_bytes(StreamGeom<LPR>::max_window_rows)));
    if (e != cudaSuccess) return e;
    const unsigned blocks = static_cast<unsigned>((A.rows + window - 1) / window);
    csr_stream_kernel<LPR><<<blocks, kThreads, smem, stream>>>(A.rows, A.nnz, A.row_ptrs, A.col_indices,
                                                               A.values, x, y, window);
    count_launches(1);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// csr_pipe_kernel<LPR, U, ROBUST>: the persistent, TMA-staged form of the row-owner
// kernel (the default when the arrays are 16-byte aligned).
//
// The grid is a small multiple of the SM count; CTA b walks row windows b,
// b + grid, ... through a ring of `stages` shared-memory buffers, each guarded
// by an mbarrier.  For a window the elected thread issues three 1-D bulk
// copies (cp.async.bulk, SASS UBLKCP): the window's row_ptrs, and the 16-byte
// aligned span of values and of col_indices that covers the window's
// contiguous non-zero range.  Nothing is staged through registers or L1 and a
// window's bytes are all in flight at once, while the previous window is
// being consumed.  Row owners (LPR lanes per row) then read value / column
// pairs from shared memory, gather x through the read-only path and
// accumulate; LPR == 1 keeps the sequential separately-rounded order, so the
// result stays bit-identical to spmv_cpu_csr.
//
// Corner cases are handled per element rather than per launch: non-zeros
// outside the staged span (a window larger than the stage capacity, or the
// last <4 non-zeros of the matrix, which a 16-byte granular copy cannot
// reach without reading past the array) are fetched from global memory, and
// so are the row_ptrs of the last window (its copy would over-read).
struct PipeStageHeader {
    int base;         // non-zero index held by slot 0 of the stage
    int staged_end;   // non-zeros [base, staged_end) are in shared memory
    int rp_staged;    // row_ptrs of the window are in shared memory
    int overflow;     // the window holds more non-zeros than a stage: cooperative multi-pass path
};

// Overflow path of csr_pipe_kernel (a window whose non-zero span does not fit a stage, e.g. a
// row-owner kernel forced onto a matrix with very long rows): the whole CTA streams the span in
// passes of 2*cap products through the stage's buffer and the row owners accumulate across
// passes.  Per row the products are still added in index order, so LPR == 1 stays sequential.
// Kept out of line so that its registers do not burden the common path.
template <int LPR>
__device__ __noinline__ void pipe_overflow_window(int nr, int r0, int rows_per_group, const int* __restrict__ row_ptrs,
                                                  const int* __restrict__ col_indices, const float* __restrict__ values,
                                                  const float* __restrict__ x, float* __restrict__ y, int* s_rp,
                                                  bool rp_staged, float* s_prod, float* s_acc, int prod_cap) {
    // running sums live in shared memory (s_acc[row]), not registers: this path must not raise
    // the register count of the kernel it is called from
    constexpr int kGroups = kThreads / LPR;
    const int tid = threadIdx.x, group = tid / LPR, lane = tid % LPR;
    if (!rp_staged) {
        for (int i = tid; i <= nr; i += kThreads) s_rp[i] = row_ptrs[r0 + i];
    }
    for (int i = tid; i < nr * LPR; i += kThreads) s_acc[i] = 0.0f;  // one slot per (row, lane)
    __syncthreads();
    const int n0 = s_rp[0], n1 = s_rp[nr];
    for (int base = n0; base < n1; base += prod_cap) {
        const int hi = min(base + prod_cap, n1);
        for (int j = base + tid; j < hi; j += kThreads)
            s_prod[j - base] = __fmul_rn(dev::ld_stream_f(values + j), dev::ld_x(x + dev::ld_stream_i(col_indices + j)));
        __syncthreads();
        for (int i = 0; i < rows_per_group; ++i) {
            const int r = group + i * kGroups;
            if (r < nr) {
                const int a = max(s_rp[r], base), b = min(s_rp[r + 1], hi);
                if (a < b) {
                    float t = s_acc[r * LPR + lane];
                    for (int j = a + lane; j < b; j += LPR) t = __fadd_rn(t, s_prod[j - base]);
                    s_acc[r * LPR + lane] = t;
                }
            }
        }
        __syncthreads();
    }
    for (int i = 0; i < rows_per_group; ++i) {
        const int r = group + i * kGroups;
        float t = r < nr ? s_acc[r * LPR + lane] : 0.0f;
#pragma unroll
        for (int d = LPR / 2; d > 0; d >>= 1) t += __shfl_down_sync(0xffffffffu, t, d, LPR);
        if (lane == 0 && r < nr) y[r0 + r] = t;
    }
}

// ROBUST = true adds the cooperative overflow path (a few registers and ~5 % on regular
// matrices); ROBUST = false stages what fits and lets row owners fetch the rest from global,
// which is only acceptable when no row comes near the stage capacity.  The launcher picks by the
// matrix's longest row (cached per device array, see longest_row_cached()); both are correct for
// any input.
template <int LPR, int U, bool ROBUST>
__global__ void __launch_bounds__(kThreads)
csr_pipe_kernel(int rows, int nnz, const int* __restrict__ row_ptrs, const int* __restrict__ col_indices,
                const float* __restrict__ values, const float* __restrict__ x, float* __restrict__ y,
                int window_rows, int rows_per_group, int cap, int stages) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);  // [stages] (<= 16)
    unsigned char* ring = smem_raw + 128;
    const size_t stage_bytes = sizeof(PipeStageHeader) + static_cast<size_t>(window_rows + 4) * 4 +
                               static_cast<size_t>(cap) * 8;
    constexpr int kGroups = kThreads / LPR;
    // U = gathers per row and batch (template parameter: 4, 6 or 8)
    const int tid = threadIdx.x;
    const int group = tid / LPR;
    const int lane = tid % LPR;
    const int num_windows = (rows + window_rows - 1) / window_rows;

    auto stage_header = [&](int s) { return reinterpret_cast<PipeStageHeader*>(ring + s * stage_bytes); };
    auto stage_rp = [&](int s) { return reinterpret_cast<int*>(ring + s * stage_bytes + sizeof(PipeStageHeader)); };
    auto stage_val = [&](int s) { return reinterpret_cast<float*>(stage_rp(s) + window_rows + 4); };
    auto stage_col = [&](int s) { return reinterpret_cast<int*>(stage_val(s) + cap); };

    // thread 0 only; n0 / n1 = first / one-past-last non-zero of the window
    auto issue = [&](int w, int s, int n0, int n1) {
        const int r0 = w * window_rows;
        const int base = n0 & ~3;
        int end = min((n1 + 3) & ~3, nnz & ~3);
        const bool overflow = ROBUST && end - base > cap;  // does not fit a stage: nothing is staged
        if (overflow) end = base;
        end = min(end, base + cap);
        end = max(end, base);
        const bool rp_ok = r0 + window_rows + 4 <= rows + 1;
        PipeStageHeader* h = stage_header(s);
        h->base = base;
        h->staged_end = end;
        h->rp_staged = rp_ok ? 1 : 0;
        h->overflow = overflow ? 1 : 0;
        const uint32_t nz_bytes = static_cast<uint32_t>(end - base) * 4u;
        const uint32_t rp_bytes = rp_ok ? static_cast<uint32_t>(window_rows + 4) * 4u : 0u;
        dev::mbar_arrive_expect_tx(bars + s, 2u * nz_bytes + rp_bytes);
        if (rp_bytes) dev::tma_bulk_g2s(stage_rp(s), row_ptrs + r0, rp_bytes, bars + s);
        if (nz_bytes) {
            dev::tma_bulk_g2s(stage_val(s), values + base, nz_bytes, bars + s);
            dev::tma_bulk_g2s(stage_col(s), col_indices + base, nz_bytes, bars + s);
        }
    };
    auto window_bounds = [&](int w, int& n0, int& n1) {
        const int r0 = w * window_rows;
        n0 = __ldg(row_ptrs + r0);
        n1 = __ldg(row_ptrs + min(r0 + window_rows, rows));
    };

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) dev::mbar_init(bars + s, 1);
        dev::mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            const int w = blockIdx.x + s * gridDim.x;
            if (w < num_windows) {
                int n0, n1;
                window_bounds(w, n0, n1);
                issue(w, s, n0, n1);
            }
        }
    }

    int it = 0;
    for (int w = blockIdx.x; w < num_windows; w += gridDim.x, ++it) {
        const int s = it % stages;
        const uint32_t parity = (it / stages) & 1u;
        const int next = w + stages * gridDim.x;
        int next_n0 = 0, next_n1 = 0;
        if (tid == 0 && next < num_windows) window_bounds(next, next_n0, next_n1);  // latency hidden by the consume phase

        dev::mbar_wait(bars + s, parity);
        const PipeStageHeader h = *stage_header(s);
        const int* s_rp = stage_rp(s);
        const float* s_val = stage_val(s);
        const int* s_col = stage_col(s);
        const int r0 = w * window_rows;
        const int nr = min(window_rows, rows - r0);

        if (ROBUST && h.overflow) {  // CTA-uniform
            // products in the stage's value area, running sums in its column area (window * LPR <= cap)
            pipe_overflow_window<LPR>(nr, r0, rows_per_group, row_ptrs, col_indices, values, x, y, stage_rp(s),
                                      h.rp_staged != 0, stage_val(s), reinterpret_cast<float*>(stage_col(s)), cap);
        } else
        // U elements of a row are gathered per batch, so up to U independent x gathers are in
        // flight per thread (one gather latency for rows up to U*LPR long).  With several lanes
        // per row (LPR > 1) two row slots of the group are walked together, otherwise the short
        // per-lane share of a row would leave the lane with too few gathers in flight.
        if (LPR > 1) {
            for (int i = 0; i < rows_per_group; i += 2) {
                const int rA = group + i * kGroups;
                const int rB = group + (i + 1) * kGroups;
                const bool okA = rA < nr, okB = (i + 1 < rows_per_group) && rB < nr;
                int jA = 0, bA = 0, jB = 0, bB = 0;
                if (okA) {
                    jA = (h.rp_staged ? s_rp[rA] : __ldg(row_ptrs + r0 + rA)) + lane;
                    bA = h.rp_staged ? s_rp[rA + 1] : __ldg(row_ptrs + r0 + rA + 1);
                }
                if (okB) {
                    jB = (h.rp_staged ? s_rp[rB] : __ldg(row_ptrs + r0 + rB)) + lane;
                    bB = h.rp_staged ? s_rp[rB + 1] : __ldg(row_ptrs + r0 + rB + 1);
                }
                float accA = 0.0f, accB = 0.0f;
                while (jA < bA || jB < bB) {
                    float vA[U], xA[U], vB[U], xB[U];
                    int cA[U], cB[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int ja = jA + u * LPR, jb = jB + u * LPR;
                        if (ja < bA) {
                            if (ja < h.staged_end) { vA[u] = s_val[ja - h.base]; cA[u] = s_col[ja - h.base]; }
                            else { vA[u] = dev::ld_stream_f(values + ja); cA[u] = dev::ld_stream_i(col_indices + ja); }
                        }
                        if (jb < bB) {
                            if (jb < h.staged_end) { vB[u] = s_val[jb - h.base]; cB[u] = s_col[jb - h.base]; }
                            else { vB[u] = dev::ld_stream_f(values + jb); cB[u] = dev::ld_stream_i(col_indices + jb); }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        if (jA + u * LPR < bA) xA[u] = dev::ld_x(x + cA[u]);
                        if (jB + u * LPR < bB) xB[u] = dev::ld_x(x + cB[u]);
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        if (jA + u * LPR < bA) accA = __fadd_rn(accA, __fmul_rn(vA[u], xA[u]));
                        if (jB + u * LPR < bB) accB = __fadd_rn(accB, __fmul_rn(vB[u], xB[u]));
                    }
                    jA += U * LPR;
                    jB += U * LPR;
                }
#pragma unroll
                for (int d = LPR / 2; d > 0; d >>= 1) {
                    accA += __shfl_down_sync(0xffffffffu, accA, d, LPR);
                    accB += __shfl_down_sync(0xffffffffu, accB, d, LPR);
                }
                if (lane == 0 && okA) y[r0 + rA] = accA;
                if (lane == 0 && okB) y[r0 + rB] = accB;
            }
        } else
        for (int i = 0; i < rows_per_group; ++i) {
            const int r = group + i * kGroups;
            float acc = 0.0f;
            if (r < nr) {
                const int a = h.rp_staged ? s_rp[r] : __ldg(row_ptrs + r0 + r);
                const int b = h.rp_staged ? s_rp[r + 1] : __ldg(row_ptrs + r0 + r + 1);
                for (int j = a + lane; j < b; j += U * LPR) {
                    float v[U], xv[U];
                    int c[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int ju = j + u * LPR;
                        if (ju < b) {
                            if (ju < h.staged_end) {
                                v[u] = s_val[ju - h.base];
                                c[u] = s_col[ju - h.base];
                            } else {
                                v[u] = dev::ld_stream_f(values + ju);
                                c[u] = dev::ld_stream_i(col_indices + ju);
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (j + u * LPR < b) xv[u] = dev::ld_x(x + c[u]);
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (j + u * LPR < b) acc = __fadd_rn(acc, __fmul_rn(v[u], xv[u]));
                }
            }
#pragma unroll
            for (int d = LPR / 2; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d, LPR);
            if (lane == 0 && r < nr) y[r0 + r] = acc;
        }
        __syncthreads();  // stage s is free again
        if (tid == 0 && next < num_windows) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(next, s, next_n0, next_n1);
        }
    }
}

// ------------------------------------------------------------------------------------------
// csr_short_kernel -- SCALAR_CSR / one-lane VECTOR_CSR for matrices of SHORT rows (the reference's
// thread-per-row kernel, src/spmv_kernels.cu:168-188, and what spmv_auto_config sends the 5-point
// Laplacian of BASELINE config 2 to): the persistent TMA ring of csr_pipe_kernel (row_ptrs window +
// aligned value / column spans per stage) consumed by ROW OWNERS with nothing else in the loop.
// ncu of csr_pipe_kernel<1,6,false> on config 2 (profiles/r1_csr_pipe_c2.md) showed it issue-bound:
// 45 thread instructions per non-zero (a "staged or global?" branch per element) and 63 registers =
// 4 CTAs per SM.  Here a window is either entirely staged -- then a row costs one predicate per slot
// and ~8 instructions per non-zero, in <= 32 registers (8 CTAs = 2048 threads per SM, like the ELL
// kernel) -- or (CTA-uniform, rare: the matrix tail, a window denser than a stage) its rows are walked
// from global memory.  Per row this is spmv_cpu_csr's `sum += values[j] * x[col[j]]` front to back
// with separately rounded multiply and add (reference src/spmv_cpu.cpp:6-16) => bit-identical.
__device__ __noinline__ void short_rows_from_global(int nr, const int* __restrict__ rp, const int* __restrict__ col_indices,
                                                    const float* __restrict__ values, const float* __restrict__ x,
                                                    float* __restrict__ y) {
    for (int r = threadIdx.x; r < nr; r += kThreads) {
        const int a = __ldg(rp + r), b = __ldg(rp + r + 1);
        float acc = 0.0f;
#pragma unroll 1
        for (int j = a; j < b; ++j)
            acc = __fadd_rn(acc, __fmul_rn(dev::ld_stream_f(values + j), dev::ld_x(x + dev::ld_stream_i(col_indices + j))));
        y[r] = acc;
    }
}

// Compile-time geometry: RPT rows per thread (window = 256 * RPT rows), CAP staged non-zeros per
// stage, S stages -- every shared-memory address in the loop is then base + immediate.
template <int RPT, int CAP>
struct ShortStage {
    static constexpr int kWindow = kThreads * RPT;
    int rp[kWindow + 4];   // row_ptrs[r0 .. r0 + kWindow + 3]
    float val[CAP];        // values[base .. staged_end)
    int col[CAP];          // col_indices[base .. staged_end)
    int base;              // non-zero index held by slot 0
    int staged;            // 0: the window was not staged (matrix tail / denser than CAP)
    int pad[2];
};

template <int U, int RPT, int CAP, int S>
__global__ void __launch_bounds__(kThreads, (CAP <= 1536 ? 8 : (CAP <= 3072 ? 4 : 2)))
csr_short_kernel(int rows, int nnz, const int* __restrict__ row_ptrs, const int* __restrict__ col_indices,
                 const float* __restrict__ values, const float* __restrict__ x, float* __restrict__ y) {
    using Stage = ShortStage<RPT, CAP>;
    constexpr int kWindow = Stage::kWindow;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);  // [S]: the stage's bulk copies have landed
    Stage* ring = reinterpret_cast<Stage*>(smem_raw + 128);
    const int tid = threadIdx.x;
    const int num_windows = (rows + kWindow - 1) / kWindow;

    auto issue = [&](int w, int s, int n0, int n1) {  // thread 0 only; [n0, n1) = the window's non-zeros
        const int r0 = w * kWindow;
        const int base = n0 & ~3;
        const int end = (n1 + 3) & ~3;
        // all or nothing: the window is staged when its row_ptrs can be bulk-copied without
        // over-reading, its span fits the stage and does not reach into the unaligned matrix tail
        const bool staged = r0 + kWindow + 4 <= rows + 1 && end - base <= CAP && end <= (nnz & ~3);
        Stage& st = ring[s];
        st.base = base;
        st.staged = staged ? 1 : 0;
        const uint32_t nz_bytes = staged ? static_cast<uint32_t>(end - base) * 4u : 0u;
        const uint32_t rp_bytes = staged ? static_cast<uint32_t>(kWindow + 4) * 4u : 0u;
        dev::mbar_arrive_expect_tx(full + s, 2u * nz_bytes + rp_bytes);
        if (rp_bytes) dev::tma_bulk_g2s(st.rp, row_ptrs + r0, rp_bytes, full + s);
        if (nz_bytes) {
            dev::tma_bulk_g2s(st.val, values + base, nz_bytes, full + s);
            dev::tma_bulk_g2s(st.col, col_indices + base, nz_bytes, full + s);
        }
    };

    if (tid == 0) {
        for (int s = 0; s < S; ++s) dev::mbar_init(full + s, 1);
        dev::mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            const int w = blockIdx.x + s * gridDim.x;
            if (w < num_windows) issue(w, s, __ldg(row_ptrs + w * kWindow), __ldg(row_ptrs + min((w + 1) * kWindow, rows)));
        }
    }

    int s = 0;
    uint32_t parity = 0;
    for (int w = blockIdx.x; w < num_windows; w += gridDim.x) {
        const int next = w + S * gridDim.x;
        int next_n0 = 0, next_n1 = 0;
        if (tid == 0 && next < num_windows) {  // a DRAM round trip, hidden by this window's consume phase
            next_n0 = __ldg(row_ptrs + next * kWindow);
            next_n1 = __ldg(row_ptrs + min((next + 1) * kWindow, rows));
        }
        dev::mbar_wait(full + s, parity);
        const Stage& st = ring[s];
        const int r0 = w * kWindow;
        const int nr = min(kWindow, rows - r0);
        if (st.staged) {
            const int base = st.base;
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                const int r = tid + i * kThreads;
                if (r < nr) {
                    const int a = st.rp[r] - base;   // stage slot of the row's first non-zero
                    const int len = st.rp[r + 1] - base - a;
                    const float* pv = st.val + a;
                    const int* pc = st.col + a;
                    float acc = 0.0f;
                    for (int j = 0; j < len; j += U) {
                        int c[U];
                        float xv[U];
#pragma unroll
                        for (int u = 0; u < U; ++u)
                            if (j + u < len) c[u] = pc[j + u];
#pragma unroll
                        for (int u = 0; u < U; ++u)
                            if (j + u < len) xv[u] = dev::ld_x(x + c[u]);
#pragma unroll
                        for (int u = 0; u < U; ++u)
                            if (j + u < len) acc = __fadd_rn(acc, __fmul_rn(pv[j + u], xv[u]));
                    }
                    y[r0 + r] = acc;
                }
            }
        } else {  // not staged: the same rows, the same order, from global memory
            short_rows_from_global(nr, row_ptrs + r0, col_indices, values, x, y + r0);
        }
        // A CTA-wide barrier frees the stage.  (Measured alternative: per-stage `empty` mbarriers that
        // only thread 0 waits on -- 0.168 ms against 0.144 ms on config 2: the warps drift apart and
        // the refill waits for the slowest anyway.)
        __syncthreads();
        if (tid == 0 && next < num_windows) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(next, s, next_n0, next_n1);
        }
        if (++s == S) {
            s = 0;
            parity ^= 1u;
        }
    }
}

// window = groups * rows_per_group rows holding about 1.5 K non-zeros; cap = stage capacity
template <int LPR>
void pipe_geometry(const CsrView& A, int& rpg, int& cap) {
    constexpr int groups = kThreads / LPR;
    const double avg = static_cast<double>(A.nnz) / A.rows;
    // measured on config 2 (profiles/r1_ell_tuning.md): ~1.5 K non-zeros per window for one lane per row,
    // ~2.5 K when lanes share rows (two row slots are walked together there)
    rpg = static_cast<int>((LPR == 1 ? 1536.0 : 2560.0) / (avg * groups) + 0.5);
    static const int env_rpg = env_int("SPMV_B200_CSR_RPG", 0);
    if (env_rpg > 0) rpg = env_rpg;
    rpg = rpg < 1 ? 1 : (rpg > 8 ? 8 : rpg);
    const int window = groups * rpg;
    cap = static_cast<int>(1.125 * avg * window) + 32;
    if (cap < kThreads * rpg) cap = kThreads * rpg;  // the overflow path keeps window * LPR running sums there
    cap = (cap + 127) / 128 * 128;
}

// Longest row of a device CSR, computed once per (row_ptrs array, shape) with one pass over
// row_ptrs and remembered.  It only steers the choice between two correct kernels, so a stale
// entry (the array was rewritten in place) costs speed, never correctness.
std::mutex& longest_mu() { static std::mutex mu; return mu; }
std::unordered_map<unsigned long long, int>& longest_cache() { static std::unordered_map<unsigned long long, int> c; return c; }
unsigned long long longest_key(const int* d_row_ptrs, int rows, int nnz) {
    return (reinterpret_cast<uintptr_t>(d_row_ptrs) * 0x9E3779B97F4A7C15ull) ^ (static_cast<unsigned long long>(rows) << 32) ^
           static_cast<unsigned>(nnz);
}

int longest_row_cached(const CsrView& A, cudaStream_t stream) {
    std::mutex& mu = longest_mu();
    std::unordered_map<unsigned long long, int>& cache = longest_cache();
    const unsigned long long key = longest_key(A.row_ptrs, A.rows, A.nnz);
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) return it->second;
    }
    // the measurement below synchronises the stream, which would invalidate an ongoing capture: while
    // capturing, an unknown matrix takes the robust kernel (correct for any row length) and is not cached
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &capturing) != cudaSuccess) cudaGetLastError();
    if (capturing != cudaStreamCaptureStatusNone) return 0x7fffffff;
    int* d_max = nullptr;
    int longest = 0x7fffffff;  // unknown -> robust kernel
    if (cudaMalloc(&d_max, sizeof(int)) == cudaSuccess) {
        cudaMemsetAsync(d_max, 0, sizeof(int), stream);
        if (launch_max_row_len(A, d_max, stream) == cudaSuccess &&
            cudaMemcpyAsync(&longest, d_max, sizeof(int), cudaMemcpyDeviceToHost, stream) == cudaSuccess &&
            cudaStreamSynchronize(stream) == cudaSuccess) {
            std::lock_guard<std::mutex> lock(mu);
            if (cache.size() > 4096) cache.clear();
            cache[key] = longest;
        } else {
            cudaGetLastError();
            longest = 0x7fffffff;
        }
        cudaFree(d_max);
    } else {
        cudaGetLastError();
    }
    return longest;
}

template <int LPR, int U, bool ROBUST>
cudaError_t launch_pipe_lpr_u(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    constexpr int groups = kThreads / LPR;
    int rpg, cap;
    pipe_geometry<LPR>(A, rpg, cap);
    const int window = groups * rpg;
    static const int env_stages = env_int("SPMV_B200_CSR_STAGES", 0);
    static const int env_ctas = env_int("SPMV_B200_CSR_CTAS_PER_SM", 0);
    const int stages = env_stages > 1 ? (env_stages > 16 ? 16 : env_stages) : 2;
    const size_t stage_bytes = sizeof(PipeStageHeader) + static_cast<size_t>(window + 4) * 4 + static_cast<size_t>(cap) * 8;
    const size_t smem = 128 + stages * stage_bytes;
    if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;  // caller falls back
    cudaError_t e = cudaFuncSetAttribute(csr_pipe_kernel<LPR, U, ROBUST>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    // A persistent grid must not exceed what is co-resident (registers AND shared memory),
    // otherwise the surplus CTAs only start when the first wave has finished.
    int fit = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, csr_pipe_kernel<LPR, U, ROBUST>, kThreads, smem);
    if (e != cudaSuccess) return e;
    if (fit < 1) return cudaErrorInvalidConfiguration;
    const int ctas_per_sm = (env_ctas > 0 && env_ctas < fit) ? env_ctas : fit;
    int sms = 148, dev_id = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
    const int num_windows = (A.rows + window - 1) / window;
    int blocks = sms * ctas_per_sm;
    if (blocks > num_windows) blocks = num_windows;
    csr_pipe_kernel<LPR, U, ROBUST><<<blocks, kThreads, smem, stream>>>(A.rows, A.nnz, A.row_ptrs, A.col_indices, A.values, x, y,
                                                             window, rpg, cap, stages);
    count_launches(1);
    return cudaGetLastError();
}

// gathers per batch: enough to cover an average row of the group's lanes in one batch
template <int LPR>
cudaError_t launch_pipe_lpr(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    static const int env_u = env_int("SPMV_B200_CSR_U", 0);
    const double per_lane = static_cast<double>(A.nnz) / A.rows / LPR;
    int u = per_lane <= 4.0 ? 4 : (per_lane <= 6.0 ? 6 : 8);
    if (env_u > 0) u = env_u;
    // a row that takes more than half a stage means windows that do not fit: robust variant
    int rpg, cap;
    pipe_geometry<LPR>(A, rpg, cap);
    static const int env_robust = env_int("SPMV_B200_CSR_ROBUST", -1);
    const bool robust = env_robust >= 0 ? env_robust != 0 : longest_row_cached(A, stream) > cap / 2;
    if (robust) {
        if (u <= 4) return launch_pipe_lpr_u<LPR, 4, true>(A, x, y, stream);
        if (u <= 6) return launch_pipe_lpr_u<LPR, 6, true>(A, x, y, stream);
        return launch_pipe_lpr_u<LPR, 8, true>(A, x, y, stream);
    }
    if (u <= 4) return launch_pipe_lpr_u<LPR, 4, false>(A, x, y, stream);
    if (u <= 6) return launch_pipe_lpr_u<LPR, 6, false>(A, x, y, stream);
    return launch_pipe_lpr_u<LPR, 8, false>(A, x, y, stream);
}

template <int U, int RPT, int CAP>
cudaError_t launch_short_as(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    constexpr int S = 2;  // ring depth: deeper rings leave fewer CTAs per SM (measured: 3 stages 0.166 ms against 0.144 ms)
    auto kernel = csr_short_kernel<U, RPT, CAP, S>;
    const size_t smem = 128 + S * sizeof(ShortStage<RPT, CAP>);
    static const int env_ctas = env_int("SPMV_B200_CSR_CTAS_PER_SM", 0);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    int fit = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, kernel, kThreads, smem);
    if (e != cudaSuccess) return e;
    if (fit < 1) return cudaErrorInvalidConfiguration;
    const int ctas_per_sm = (env_ctas > 0 && env_ctas < fit) ? env_ctas : fit;
    int sms = 148, dev_id = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
    constexpr int window = kThreads * RPT;
    const int num_windows = (A.rows + window - 1) / window;
    int blocks = sms * ctas_per_sm;
    if (blocks > num_windows) blocks = num_windows;
    kernel<<<blocks, kThreads, smem, stream>>>(A.rows, A.nnz, A.row_ptrs, A.col_indices, A.values, x, y);
    count_launches(1);
    return cudaGetLastError();
}

// Geometry by the average row length: a window should hold 1.3-1.5 K non-zeros (measured on config 2:
// 1024 / 1536 / 2560 per window -> 0.145 / 0.144 / 0.155 ms) with 12.5 % head-room in the stage.
cudaError_t launch_short(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    const double avg = static_cast<double>(A.nnz) / A.rows;
    if (avg <= 2.6) return launch_short_as<4, 2, 1536>(A, x, y, stream);    // 512-row windows
    if (avg <= 5.2) return launch_short_as<6, 1, 1536>(A, x, y, stream);    // 256-row windows, 8 CTAs per SM
    return launch_short_as<8, 1, 3072>(A, x, y, stream);                    // avg <= 10.5: 4 CTAs per SM
    // (a 5120-entry stage for avg <= 16 leaves 2 CTAs per SM and loses to the general ring: 13-point stencil
    //  0.109 against 0.092 ms, scripts/time_mid.py)
}

// Short rows only: a row is walked by one thread, and a window that does not fit a stage is walked
// from global memory by 256 threads -- both fine while no row is long.
bool short_eligible(const CsrView& A, cudaStream_t stream) {
    static const int mode = env_int("SPMV_B200_CSR_SHORT", -1);  // 0 off, 1 forced, -1 by structure
    if (mode == 0) return false;
    if (mode == 1) return true;
    const double avg = static_cast<double>(A.nnz) / A.rows;
    if (avg > 10.5) return false;  // launch_short's largest stage
    // UNIFORM rows only (stencils, meshes, banded systems: longest <= avg + 1.5): there the lean loop wins
    // (config 2: 0.129 against 0.164 ms).  On rows of random length 0 .. 2 avg with random columns it LOSES to
    // the general ring (scripts/time_mid.py, 4 M rows: avg 5 0.159 against 0.103 ms, avg 8 0.250 against
    // 0.158 ms): a warp waits for its longest row in batches of U dependent gathers, and 32 registers leave
    // fewer gathers in flight per thread than the general ring's 63.
    return static_cast<double>(longest_row_cached(A, stream)) <= avg + 1.5;
}

bool pipe_eligible(const CsrView& A) {
    static const int disable = env_int("SPMV_B200_CSR_NO_PIPE", 0);
    const uintptr_t bits = reinterpret_cast<uintptr_t>(A.values) | reinterpret_cast<uintptr_t>(A.col_indices) |
                           reinterpret_cast<uintptr_t>(A.row_ptrs);
    return !disable && (bits & 15u) == 0;
}

template <int LPR>
cudaError_t launch_best_lpr(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    if (pipe_eligible(A)) {
        if (LPR == 1 && short_eligible(A, stream)) {
            const cudaError_t e = launch_short(A, x, y, stream);
            if (e != cudaErrorInvalidConfiguration) return e;
        }
        const cudaError_t e = launch_pipe_lpr<LPR>(A, x, y, stream);
        if (e != cudaErrorInvalidConfiguration) return e;
    }
    return launch_stream_lpr<LPR>(A, x, y, stream);
}

}  // namespace

// csr_to_gpu knows the host row_ptrs: it seeds the longest-row cache so that the first stream-ordered
// SCALAR / VECTOR launch on an uploaded matrix neither allocates nor synchronises (the lazy device pass
// remains for device arrays supplied by the caller); csr_free_gpu / csr_to_gpu drop the entry.
void seed_longest_row(const int* d_row_ptrs, int rows, int nnz, int longest) {
    if (!d_row_ptrs) return;
    std::lock_guard<std::mutex> lock(longest_mu());
    auto& cache = longest_cache();
    if (cache.size() > 4096) cache.clear();
    cache[longest_key(d_row_ptrs, rows, nnz)] = longest;
}
void forget_longest_row(const int* d_row_ptrs, int rows, int nnz) {
    if (!d_row_ptrs) return;
    std::lock_guard<std::mutex> lock(longest_mu());
    longest_cache().erase(longest_key(d_row_ptrs, rows, nnz));
}

cudaError_t launch_csr_stream(const CsrView& A, const float* x, float* y, int lanes_per_row,
                              cudaStream_t stream) {
    if (A.rows <= 0) return cudaSuccess;
    if (A.nnz <= 0) {
        zero_rows_kernel<<<(A.rows + 255) / 256, 256, 0, stream>>>(A.rows, y);
        count_launches(1);
        return cudaGetLastError();
    }
    switch (lanes_per_row) {
        case 1:  return launch_best_lpr<1>(A, x, y, stream);
        case 2:  return launch_best_lpr<2>(A, x, y, stream);
        case 4:  return launch_best_lpr<4>(A, x, y, stream);
        case 8:  return launch_best_lpr<8>(A, x, y, stream);
        case 16: return launch_best_lpr<16>(A, x, y, stream);
    }
    switch (lanes_per_row) {
        case 1:  return launch_stream_lpr<1>(A, x, y, stream);
        case 2:  return launch_stream_lpr<2>(A, x, y, stream);
        case 4:  return launch_stream_lpr<4>(A, x, y, stream);
        case 8:  return launch_stream_lpr<8>(A, x, y, stream);
        default: return launch_stream_lpr<16>(A, x, y, stream);
    }
}

cudaError_t launch_csr_warp_per_row(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    if (A.rows <= 0) return cudaSuccess;
    const long long threads = static_cast<long long>(A.rows) * 32;
    const unsigned blocks = static_cast<unsigned>((threads + kThreads - 1) / kThreads);
    csr_warp_row_kernel<<<blocks, kThreads, 0, stream>>>(A.rows, A.row_ptrs, A.col_indices, A.values, x, y);
    count_launches(1);
    return cudaGetLastError();
}

// lanes per row for VECTOR_CSR from the average row length:
// <20 -> 1, <32 -> 8, <64 -> 16, else a full warp.
// One lane per row IS the row-owner pipeline of SCALAR_CSR (sequential order): on rows this short
// sharing a row between lanes only adds shuffles -- config 2 (5 per row): 0.165 ms against 0.183 ms
// with two lanes.  The selector only sends matrices with max <= 10 * (min + 1) here, so no lane is
// left alone with a long row.  SPMV_B200_VECTOR_LANES forces a width (A/B timing).
int vector_lanes_for(int rows, int nnz) {
    static const int forced = env_int("SPMV_B200_VECTOR_LANES", 0);
    if (forced == 1 || forced == 2 || forced == 4 || forced == 8 || forced == 16 || forced == 32) return forced;
    const double avg = rows > 0 ? static_cast<double>(nnz) / rows : 0.0;
    // measured on 4 M-row matrices (scripts/time_mid.py), one lane against the old choice of 2 / 4 / 8 lanes:
    // 7-point stencil 0.052 / 0.062 ms, 9-point 0.060 / 0.088, 13-point 0.092 / 0.116, random rows avg 8
    // 0.158 / 0.258, avg 12 0.228 / 0.247, avg 16 0.302 / 0.313, avg 24 0.745 / 0.478 -> one lane below 20
    if (avg < 20.0) return 1;
    if (avg < 32.0) return 8;
    if (avg < 64.0) return 16;
    return 32;
}

cudaError_t launch_csr_vector(const CsrView& A, const float* x, float* y, cudaStream_t stream) {
    const int lanes = vector_lanes_for(A.rows, A.nnz);
    if (lanes == 32) return launch_csr_warp_per_row(A, x, y, stream);
    return launch_csr_stream(A, x, y, lanes, stream);
}

}  // namespace b200
}  // namespace spmv
