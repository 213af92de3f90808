// ell_kernels.cu -- column-major ELL SpMV for sm_100a.
//
// Replaces spmv_ell_kernel (reference src/spmv_kernels.cu:191-213): there one
// thread owns one row and issues 32-bit loads.  Here one thread owns RPT
// ADJACENT rows so every slice k is read with one 128-bit (RPT=4) or 64-bit
// (RPT=2) load of values and one of col_indices -- a warp covers 128 rows and
// reads 512 contiguous bytes per array per slice.  Matrix data streams through
// ld.global.nc.L1::no_allocate; x is gathered through the read-only path and
// stays L1/L2 resident; y leaves with one vector store.
//
// Per row the products are accumulated in slice order k = 0..W-1 with a
// separately rounded multiply and add (__fmul_rn/__fadd_rn), i.e. exactly the
// operation order of spmv_cpu_ell (reference src/spmv_cpu.cpp:18-32): the
// result is bit-identical to the reference's CPU path.
//
// Roofline: HBM.  Algorithmic bytes per launch = 8*rows*W + 4*cols + 4*rows
// (reference src/bandwidth.cpp:66-75).
#include "device_utils.cuh"
#include "internal.hpp"

namespace spmv {
namespace b200 {
namespace {

constexpr int kEllThreads = 256;
constexpr int kEllBatch = 4;  // slices in flight per thread

template <int RPT> struct VecLoad;
template <> struct VecLoad<4> {
    static __device__ __forceinline__ void load(const float* v, const int* c, float (&fv)[4], int (&ic)[4]) {
        const float4 a = dev::ld_stream_f4(v);
        const int4 b = dev::ld_stream_i4(c);
        fv[0] = a.x; fv[1] = a.y; fv[2] = a.z; fv[3] = a.w;
        ic[0] = b.x; ic[1] = b.y; ic[2] = b.z; ic[3] = b.w;
    }
    static __device__ __forceinline__ void store(float* y, const float (&s)[4]) {
        dev::st_stream_f4(y, make_float4(s[0], s[1], s[2], s[3]));
    }
};
template <> struct VecLoad<2> {
    static __device__ __forceinline__ void load(const float* v, const int* c, float (&fv)[2], int (&ic)[2]) {
        const float2 a = dev::ld_stream_f2(v);
        const int2 b = dev::ld_stream_i2(c);
        fv[0] = a.x; fv[1] = a.y;
        ic[0] = b.x; ic[1] = b.y;
    }
    static __device__ __forceinline__ void store(float* y, const float (&s)[2]) {
        dev::st_stream_f2(y, make_float2(s[0], s[1]));
    }
};
template <> struct VecLoad<1> {
    static __device__ __forceinline__ void load(const float* v, const int* c, float (&fv)[1], int (&ic)[1]) {
        fv[0] = dev::ld_stream_f(v);
        ic[0] = dev::ld_stream_i(c);
    }
    static __device__ __forceinline__ void store(float* y, const float (&s)[1]) { y[0] = s[0]; }
};

// rows % RPT == 0 and all pointers aligned to 4*RPT bytes (checked by the launcher)
template <int RPT>
__global__ void __launch_bounds__(kEllThreads)
ell_slice_kernel(int rows, int width, const int* __restrict__ col_indices,
                 const float* __restrict__ values, const float* __restrict__ x,
                 float* __restrict__ y, unsigned long long* __restrict__ nnz_counter) {
    const long long row0 = (static_cast<long long>(blockIdx.x) * kEllThreads + threadIdx.x) * RPT;
    unsigned live = 0;
    if (row0 < rows) {
        float acc[RPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i) acc[i] = 0.0f;

        const size_t stride = static_cast<size_t>(rows);
        const float* vp = values + row0;
        const int* cp = col_indices + row0;

        for (int k0 = 0; k0 < width; k0 += kEllBatch) {
            float fv[kEllBatch][RPT];
            int ic[kEllBatch][RPT];
            float xv[kEllBatch][RPT];
            // issue every load of the batch before the first use
#pragma unroll
            for (int b = 0; b < kEllBatch; ++b) {
                if (k0 + b < width) VecLoad<RPT>::load(vp + (k0 + b) * stride, cp + (k0 + b) * stride, fv[b], ic[b]);
            }
#pragma unroll
            for (int b = 0; b < kEllBatch; ++b) {
                if (k0 + b < width) {
#pragma unroll
                    for (int i = 0; i < RPT; ++i) xv[b][i] = ic[b][i] >= 0 ? dev::ld_x(x + ic[b][i]) : 0.0f;
                }
            }
#pragma unroll
            for (int b = 0; b < kEllBatch; ++b) {
                if (k0 + b < width) {
#pragma unroll
                    for (int i = 0; i < RPT; ++i) {
                        if (ic[b][i] >= 0) {  // padding slots are skipped, not multiplied
                            acc[i] = __fadd_rn(acc[i], __fmul_rn(fv[b][i], xv[b][i]));
                            ++live;
                        }
                    }
                }
            }
        }
        VecLoad<RPT>::store(y + row0, acc);
    }
    if (nnz_counter != nullptr) {  // true (non-padding) entry count for the GFLOPS figure
        live = dev::warp_sum(live);
        if ((threadIdx.x & 31) == 0 && live) atomicAdd(nnz_counter, static_cast<unsigned long long>(live));
    }
}

template <int RPT>
cudaError_t launch_rpt(int rows, int width, const int* ci, const float* va, const float* x, float* y,
                       unsigned long long* counter, cudaStream_t stream) {
    const long long threads = (static_cast<long long>(rows) + RPT - 1) / RPT;
    const unsigned blocks = static_cast<unsigned>((threads + kEllThreads - 1) / kEllThreads);
    ell_slice_kernel<RPT><<<blocks, kEllThreads, 0, stream>>>(rows, width, ci, va, x, y, counter);
    count_launches(1);
    return cudaGetLastError();
}

bool all_aligned(const void* a, const void* b, const void* c, unsigned bytes) {
    const uintptr_t m = bytes - 1;
    return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
             reinterpret_cast<uintptr_t>(c)) & m) == 0;
}

__global__ void zero_rows_kernel(int rows, float* __restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rows) y[i] = 0.0f;
}

// ---------------------------------------------------------------------------
// TMA-staged variant.  A CTA owns a window of RPT*256 consecutive rows.  One
// elected thread issues, for every slice k of the pass, one 1-D bulk copy
// (cp.async.bulk, SASS UBLKCP) of the window's values and one of its
// col_indices into shared memory and arms a single mbarrier with the total
// byte count: the whole window (2 * KS * rows * 4 bytes, 40 KB for the
// Laplacian) is in flight at once with no register staging and without
// passing through L1.  Row owners then read their slots from shared memory
// (stride-1 across a warp: conflict-free), gather x through the read-only
// path (a warp's rows are adjacent, so a stencil gather touches one or two
// lines) and accumulate in slice order with separately rounded multiply/add,
// exactly like ell_slice_kernel.  Thread t owns rows t, t+256, ...
// Needs rows % 4 == 0 and 16-byte aligned arrays (checked by the launcher).
template <int RPT>
__global__ void __launch_bounds__(kEllThreads)
ell_tma_kernel(int rows, int width, int slices_per_pass, const int* __restrict__ col_indices,
               const float* __restrict__ values, const float* __restrict__ x, float* __restrict__ y,
               unsigned long long* __restrict__ nnz_counter) {
    constexpr int kWindow = RPT * kEllThreads;
    extern __shared__ __align__(16) unsigned char ell_smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(ell_smem);
    float* s_val = reinterpret_cast<float*>(ell_smem + 16);                       // [slices_per_pass][kWindow]
    int* s_col = reinterpret_cast<int*>(ell_smem + 16) + slices_per_pass * kWindow;  // [slices_per_pass][kWindow]

    const int tid = threadIdx.x;
    const long long r0 = static_cast<long long>(blockIdx.x) * kWindow;
    const int nr = static_cast<int>(min(static_cast<long long>(kWindow), rows - r0));  // multiple of 4
    const size_t stride = static_cast<size_t>(rows);

    if (tid == 0) {
        dev::mbar_init(bar, 1);
        dev::mbar_fence_init();
    }
    __syncthreads();

    float acc[RPT];
#pragma unroll
    for (int i = 0; i < RPT; ++i) acc[i] = 0.0f;
    unsigned live = 0;
    uint32_t parity = 0;

    for (int k0 = 0; k0 < width; k0 += slices_per_pass) {
        const int ks = min(slices_per_pass, width - k0);
        if (tid == 0) {
            const uint32_t slice_bytes = static_cast<uint32_t>(nr) * sizeof(float);
            dev::mbar_arrive_expect_tx(bar, 2u * ks * slice_bytes);
            for (int k = 0; k < ks; ++k) {
                const size_t off = (k0 + k) * stride + static_cast<size_t>(r0);
                dev::tma_bulk_g2s(s_val + k * kWindow, values + off, slice_bytes, bar);
                dev::tma_bulk_g2s(s_col + k * kWindow, col_indices + off, slice_bytes, bar);
            }
        }
        dev::mbar_wait(bar, parity);
        parity ^= 1u;

#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int r = tid + i * kEllThreads;
            if (r < nr) {
                float a = acc[i];
#pragma unroll 5
                for (int k = 0; k < ks; ++k) {
                    const int c = s_col[k * kWindow + r];
                    if (c >= 0) {  // padding slots are skipped, not multiplied
                        a = __fadd_rn(a, __fmul_rn(s_val[k * kWindow + r], dev::ld_x(x + c)));
                        ++live;
                    }
                }
                acc[i] = a;
            }
        }
        if (k0 + slices_per_pass < width) {
            __syncthreads();  // every row owner is done with this pass before the buffers are refilled
            if (tid == 0) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
    }
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const int r = tid + i * kEllThreads;
        if (r < nr) y[r0 + r] = acc[i];
    }
    if (nnz_counter != nullptr) {
        live = dev::warp_sum(live);
        if ((tid & 31) == 0 && live) atomicAdd(nnz_counter, static_cast<unsigned long long>(live));
    }
}

constexpr int kEllMaxSlicesPerPass = 5;

template <int RPT>
cudaError_t launch_tma(int rows, int width, const int* ci, const float* va, const float* x, float* y,
                       unsigned long long* counter, cudaStream_t stream) {
    constexpr int kWindow = RPT * kEllThreads;
    const int slices = width < kEllMaxSlicesPerPass ? width : kEllMaxSlicesPerPass;
    const size_t smem = 16 + static_cast<size_t>(slices) * kWindow * 8;
    cudaError_t e = cudaFuncSetAttribute(ell_tma_kernel<RPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(16 + kEllMaxSlicesPerPass * kWindow * 8));
    if (e != cudaSuccess) return e;
    const unsigned blocks = static_cast<unsigned>((static_cast<long long>(rows) + kWindow - 1) / kWindow);
    ell_tma_kernel<RPT><<<blocks, kEllThreads, smem, stream>>>(rows, width, slices, ci, va, x, y, counter);
    count_launches(1);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Persistent, multi-stage form of the TMA-staged kernel (width <= 8): the grid
// is a small multiple of the SM count, CTA b walks windows b, b + grid, ...
// through a ring of `stages` shared-memory buffers, each guarded by its own
// mbarrier.  While the row owners consume window i, the bulk copies of windows
// i+1 .. i+stages-1 are already in flight, so an SM always has
// ctas_per_sm * (stages-1) * width * 8 * kWindow bytes outstanding and never
// drains at CTA boundaries.
template <int RPT>
__global__ void __launch_bounds__(kEllThreads)
ell_tma_pipe_kernel(int rows, int width, int stages, const int* __restrict__ col_indices,
                    const float* __restrict__ values, const float* __restrict__ x, float* __restrict__ y,
                    unsigned long long* __restrict__ nnz_counter, int row_lo, int row_hi) {
    // rows = slot stride of the column-major arrays (the whole matrix); this launch covers rows
    // [row_lo, row_hi) (the whole matrix, or one row chunk of the pipelined host-buffer call)
    constexpr int kWindow = RPT * kEllThreads;
    extern __shared__ __align__(16) unsigned char ell_smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(ell_smem);              // [stages] (<= 16)
    unsigned char* buffers = ell_smem + 128;
    const size_t stage_bytes = static_cast<size_t>(width) * kWindow * 8;  // values then col_indices

    const int tid = threadIdx.x;
    const size_t stride = static_cast<size_t>(rows);
    const int num_windows = static_cast<int>((static_cast<long long>(row_hi - row_lo) + kWindow - 1) / kWindow);

    auto issue = [&](int window, int stage) {  // thread 0 only
        const long long r0 = row_lo + static_cast<long long>(window) * kWindow;
        const int nr = static_cast<int>(min(static_cast<long long>(kWindow), row_hi - r0));
        const uint32_t slice_bytes = static_cast<uint32_t>(nr) * sizeof(float);
        float* s_val = reinterpret_cast<float*>(buffers + stage * stage_bytes);
        int* s_col = reinterpret_cast<int*>(s_val + width * kWindow);
        dev::mbar_arrive_expect_tx(bars + stage, 2u * width * slice_bytes);
        for (int k = 0; k < width; ++k) {
            const size_t off = k * stride + static_cast<size_t>(r0);
            dev::tma_bulk_g2s(s_val + k * kWindow, values + off, slice_bytes, bars + stage);
            dev::tma_bulk_g2s(s_col + k * kWindow, col_indices + off, slice_bytes, bars + stage);
        }
    };

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) dev::mbar_init(bars + s, 1);
        dev::mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            const int w = blockIdx.x + s * gridDim.x;
            if (w < num_windows) issue(w, s);
        }
    }

    unsigned live = 0;
    int it = 0;
    for (int w = blockIdx.x; w < num_windows; w += gridDim.x, ++it) {
        const int stage = it % stages;
        const uint32_t parity = (it / stages) & 1u;
        const long long r0 = row_lo + static_cast<long long>(w) * kWindow;
        const int nr = static_cast<int>(min(static_cast<long long>(kWindow), row_hi - r0));
        const float* s_val = reinterpret_cast<const float*>(buffers + stage * stage_bytes);
        const int* s_col = reinterpret_cast<const int*>(s_val + width * kWindow);
        dev::mbar_wait(bars + stage, parity);
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int r = tid + i * kEllThreads;
            if (r < nr) {
                float a = 0.0f;
#pragma unroll 5
                for (int k = 0; k < width; ++k) {
                    const int c = s_col[k * kWindow + r];
                    if (c >= 0) {
                        a = __fadd_rn(a, __fmul_rn(s_val[k * kWindow + r], dev::ld_x(x + c)));
                        ++live;
                    }
                }
                y[r0 + r] = a;
            }
        }
        __syncthreads();  // the stage is free again
        if (tid == 0) {
            const int next = w + stages * gridDim.x;
            if (next < num_windows) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue(next, stage);
            }
        }
    }
    if (nnz_counter != nullptr) {
        live = dev::warp_sum(live);
        if ((tid & 31) == 0 && live) atomicAdd(nnz_counter, static_cast<unsigned long long>(live));
    }
}

template <int RPT>
cudaError_t launch_tma_pipe(int rows, int width, const int* ci, const float* va, const float* x, float* y,
                            unsigned long long* counter, cudaStream_t stream, int row_lo = 0, int row_hi = -1) {
    if (row_hi < 0) row_hi = rows;
    constexpr int kWindow = RPT * kEllThreads;
    static const int env_stages = env_int("SPMV_B200_ELL_STAGES", 0);
    static const int env_ctas = env_int("SPMV_B200_ELL_CTAS_PER_SM", 0);
    const size_t stage_bytes = static_cast<size_t>(width) * kWindow * 8;
    // Measured on B200 (profiles/r1_ell_tuning.md): the consumer side (x gathers) needs every
    // thread slot of the SM, the ring only needs two stages -> 2 stages, as many CTAs as fit (<= 8).
    int stages = env_stages > 0 ? env_stages : 2;
    if (stages > 16) stages = 16;
    // a deeper ring than one CTA's shared memory holds is cut to what fits (W = 8, one row per thread:
    // 16 KiB per stage, so 16 stages would ask for 256 KiB)
    int dev_id = 0, optin = 0;
    cudaGetDevice(&dev_id);
    cudaError_t e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev_id);
    if (e != cudaSuccess) return e;
    const int fit_stages = static_cast<int>((static_cast<size_t>(optin) - 128) / stage_bytes);
    if (stages > fit_stages) stages = fit_stages;
    if (stages < 2) stages = 2;
    const size_t smem = 128 + stages * stage_bytes;
    e = cudaFuncSetAttribute(ell_tma_pipe_kernel<RPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    // a persistent grid must not exceed what is co-resident (registers and shared memory)
    int fit = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, ell_tma_pipe_kernel<RPT>, kEllThreads, smem);
    if (e != cudaSuccess) return e;
    if (fit < 1) fit = 1;
    const int ctas_per_sm = (env_ctas > 0 && env_ctas < fit) ? env_ctas : fit;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
    const int num_windows = static_cast<int>((static_cast<long long>(row_hi - row_lo) + kWindow - 1) / kWindow);
    if (num_windows <= 0) return cudaSuccess;
    int blocks = sms * ctas_per_sm;
    if (blocks > num_windows) blocks = num_windows;
    ell_tma_pipe_kernel<RPT><<<blocks, kEllThreads, smem, stream>>>(rows, width, stages, ci, va, x, y, counter, row_lo,
                                                                    row_hi);
    count_launches(1);
    return cudaGetLastError();
}

// 0 = automatic; 1 = register-staged kernel; 2 / 3 = TMA-staged with 4 / 2 rows per thread;
// 4 / 5 / 6 = persistent TMA pipeline with 4 / 2 / 1 rows per thread.
// (SPMV_B200_ELL_VARIANT exists for A/B timing on the device; see profiles/.)
int ell_variant_override() {
    static const int v = env_int("SPMV_B200_ELL_VARIANT", 0);
    return v;
}

}  // namespace

cudaError_t launch_ell(int rows, int width, const int* col_indices, const float* values,
                       const float* x, float* y, unsigned long long* nnz_counter, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    if (width <= 0) {  // no stored entries: y = 0
        zero_rows_kernel<<<(rows + 255) / 256, 256, 0, stream>>>(rows, y);
        count_launches(1);
        return cudaGetLastError();
    }
    if (rows % 4 == 0 && all_aligned(col_indices, values, y, 16)) {
        const int variant = ell_variant_override();
        if (variant == 1) return launch_rpt<4>(rows, width, col_indices, values, x, y, nnz_counter, stream);
        if (variant == 2) return launch_tma<4>(rows, width, col_indices, values, x, y, nnz_counter, stream);
        if (width <= 8) {
            if (variant == 4) return launch_tma_pipe<4>(rows, width, col_indices, values, x, y, nnz_counter, stream);
            if (variant == 5) return launch_tma_pipe<2>(rows, width, col_indices, values, x, y, nnz_counter, stream);
            if (variant != 3) return launch_tma_pipe<1>(rows, width, col_indices, values, x, y, nnz_counter, stream);
        }
        return launch_tma<2>(rows, width, col_indices, values, x, y, nnz_counter, stream);
    }
    if (rows % 2 == 0 && all_aligned(col_indices, values, y, 8))
        return launch_rpt<2>(rows, width, col_indices, values, x, y, nnz_counter, stream);
    return launch_rpt<1>(rows, width, col_indices, values, x, y, nnz_counter, stream);
}

// Rows [row_lo, row_hi) of the product only (row_lo % 4 == 0): one row chunk of the pipelined
// host-buffer call (host_pipeline.cu).  cudaErrorInvalidConfiguration: the matrix does not qualify
// for the TMA pipeline (alignment / width) -- the caller then multiplies the whole matrix at once.
cudaError_t launch_ell_rows(int rows, int width, const int* col_indices, const float* values, const float* x, float* y,
                            int row_lo, int row_hi, cudaStream_t stream) {
    if (rows <= 0 || row_hi <= row_lo) return cudaSuccess;
    if (width <= 0 || width > 8 || rows % 4 != 0 || row_lo % 4 != 0 || !all_aligned(col_indices, values, y, 16))
        return cudaErrorInvalidConfiguration;
    return launch_tma_pipe<1>(rows, width, col_indices, values, x, y, nullptr, stream, row_lo, row_hi);
}

}  // namespace b200
}  // namespace spmv
