// pagerank_small.cu -- the whole PageRank loop of a SMALL graph in ONE persistent, cooperative kernel.
//
// Replaces the host loop of pagerank (reference src/pagerank.cu:93-132: per iteration two PCIe copies, spmv_csr and
// three host passes) for graphs where even the fused step of pagerank.cu is launch-bound: a graph replay of the
// step (tile kernel, fix-up, reduction, dangling hand-over) plus the 24-byte download and the event the lagged stop
// rule waits for cost ~43 us per iteration at n = 4096, where the arithmetic takes 2.  Here the iterations never leave the
// device: a grid of co-resident CTAs (cooperative launch) walks the rows warp by warp -- lanes stride over a row's
// non-zeros (hub rows of small R-MAT graphs included), exact products accumulated in f64, shuffle tree, one rounding to
// fp32 --, lane 0
// applies r_new = (d*y + d*dangling/n) + (1-d)/n in the reference's operation order (src/pagerank.cu:111-114), or its
// personalized form (dev::pr_row_value), and
// accumulates sum (delta^2), sum |delta| and the next dangling mass in f64; per-CTA partials are folded in CTA order
// by EVERY CTA after one grid barrier per iteration, so every CTA takes the same stop decision (the reference's: L2
// norm of the delta < tolerance, checked every iteration, src/pagerank.cu:118-127) without a second barrier or a
// broadcast.  Deterministic: fixed row -> warp assignment, fixed reduction orders, no float atomics.
//
// Coherence: the rank vectors ping-pong between iterations and are written by other SMs, so they are read with
// ld.global.cg (L2) -- never through the non-coherent path; the matrix and the dangling bitmask are constant and go
// through ld.global.nc.
#include "device_utils.cuh"
#include "internal.hpp"

#include <cmath>

namespace spmv {
namespace b200 {
namespace {

constexpr int kSmallThreads = 512;
constexpr int kSmallWarps = kSmallThreads / 32;

struct SmallArgs {
    CsrView A;
    float damping, teleport, tolerance;  // teleport: (1 - d) / n, or 1 - d when pvec is set
    int max_iterations;
    const uint32_t* bits;  // dangling bitmask
    const float* pvec;     // normalised personalization vector [n] (PageRankStepArgs::pvec), or nullptr
    float* buf[2];         // buf[0] holds r_0 = 1/n
    const float* dsum0;    // dangling mass of r_0 (fp32, as pr_init leaves it)
    double* partials;      // [2][gridDim.x][3]
    unsigned* barrier;     // [0] arrivals, [1] generation
    float* history;        // [history_capacity] L2 residual of iteration i + 1, or nullptr
    int history_capacity;
    int* out_i;            // [0] iterations, [1] converged, [2] buffer holding the final vector
    float* out_residual;
    double* out_l1;
};

__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned blocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile unsigned* gen = bar + 1;
        const unsigned g = *gen;
        __threadfence();  // this CTA's stores before its arrival
        if (atomicAdd(bar, 1u) == blocks - 1) {
            bar[0] = 0;
            __threadfence();
            atomicAdd(bar + 1, 1u);
        } else {
            while (*gen == g) {}
        }
        __threadfence();
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kSmallThreads)
pagerank_small_kernel(SmallArgs a) {
    __shared__ double s_part[kSmallWarps][3];
    __shared__ double s_tot[3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gwarp = blockIdx.x * kSmallWarps + warp, total_warps = gridDim.x * kSmallWarps;
    const int n = a.A.rows;
    float dsum = *a.dsum0;
    int cur = 0, iters = 0, conv = 0, fin = 0;
    float residual = 0.0f;
    double l1_out = 0.0;
    for (int it = 0; it < a.max_iterations; ++it) {
        const float* r_old = a.buf[cur];
        float* r_new = a.buf[cur ^ 1];
        const float dangling_term = dev::pr_step_context(a.damping, dsum, n, a.pvec);
        double l2 = 0.0, l1 = 0.0, dang = 0.0;
        for (int row = gwarp; row < n; row += total_warps) {
            const int lo = __ldg(a.A.row_ptrs + row), hi = __ldg(a.A.row_ptrs + row + 1);
            // the row's dot product in f64 (exact products, lanes stride over the non-zeros, shuffle tree), rounded to fp32
            // once: spmv_b200_pagerank_device is the "f64 accumulators everywhere" entry point (DESIGN 5), and at these
            // sizes the extra precision is free -- the sum no longer depends on how the row is cut into lanes
            double acc = 0.0;
            int j = lo + lane;
            for (; j + 96 < hi; j += 128) {  // four independent gathers in flight per lane: a hub row is latency-bound otherwise
                const int c0 = __ldg(a.A.col_indices + j), c1 = __ldg(a.A.col_indices + j + 32);
                const int c2 = __ldg(a.A.col_indices + j + 64), c3 = __ldg(a.A.col_indices + j + 96);
                const float v0 = __ldg(a.A.values + j), v1 = __ldg(a.A.values + j + 32);
                const float v2 = __ldg(a.A.values + j + 64), v3 = __ldg(a.A.values + j + 96);
                const float x0 = __ldcg(r_old + c0), x1 = __ldcg(r_old + c1), x2 = __ldcg(r_old + c2), x3 = __ldcg(r_old + c3);
                acc += static_cast<double>(v0) * static_cast<double>(x0);
                acc += static_cast<double>(v1) * static_cast<double>(x1);
                acc += static_cast<double>(v2) * static_cast<double>(x2);
                acc += static_cast<double>(v3) * static_cast<double>(x3);
            }
            for (; j < hi; j += 32)
                acc += static_cast<double>(__ldg(a.A.values + j)) * static_cast<double>(__ldcg(r_old + __ldg(a.A.col_indices + j)));
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
            const float s = static_cast<float>(acc);
            if (lane == 0) {
                const float v = dev::pr_row_value(a.damping, s, dangling_term, a.teleport, a.pvec, row);
                __stcg(r_new + row, v);
                const double diff = static_cast<double>(v) - static_cast<double>(__ldcg(r_old + row));
                l2 += diff * diff;
                l1 += fabs(diff);
                if ((__ldg(a.bits + (row >> 5)) >> (row & 31)) & 1u) dang += static_cast<double>(v);
            }
        }
        if (lane == 0) { s_part[warp][0] = l2; s_part[warp][1] = l1; s_part[warp][2] = dang; }
        __syncthreads();
        double* mine = a.partials + (static_cast<size_t>(it & 1) * gridDim.x + blockIdx.x) * 3;
        if (threadIdx.x < 3) {
            double t = 0.0;
            for (int w = 0; w < kSmallWarps; ++w) t += s_part[w][threadIdx.x];
            __stcg(mine + threadIdx.x, t);
        }
        grid_barrier(a.barrier, gridDim.x);
        if (warp < 3) {  // every CTA folds every CTA's partials in the same order: lane l takes CTAs l, l + 32, ..., then a tree
            const double* all = a.partials + static_cast<size_t>(it & 1) * gridDim.x * 3;
            double t = 0.0;
            for (unsigned b = lane; b < gridDim.x; b += 32) t += __ldcg(all + b * 3 + warp);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
            if (lane == 0) s_tot[warp] = t;
        }
        __syncthreads();
        residual = sqrtf(static_cast<float>(s_tot[0]));  // L2 norm of the delta (reference :118)
        l1_out = s_tot[1];
        iters = it + 1;
        fin = cur ^ 1;
        if (blockIdx.x == 0 && threadIdx.x == 0 && a.history && it < a.history_capacity) a.history[it] = residual;
        if (residual < a.tolerance) { conv = 1; break; }  // reference :123-127
        dsum = static_cast<float>(s_tot[2]);
        cur ^= 1;
        __syncthreads();  // s_tot is rewritten in the next iteration
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.out_i[0] = iters;
        a.out_i[1] = conv;
        a.out_i[2] = fin;  // max_iterations == 0: buf[0], the initial vector (reference :135-139)
        *a.out_residual = residual;
        *a.out_l1 = l1_out;
    }
}

}  // namespace

// Does the one-kernel loop apply?  Small graphs only (measured, profiles/r2_small_pagerank.txt: it wins up to n = 4096,
// loses from n = 65536 on, where the merge-path step -- balanced over all SMs, hub-column / segmented plans -- takes over).  SPMV_B200_PR_SMALL=0 disables it, =2 forces it.
bool pagerank_small_applies(int n, int nnz) {
    static const int mode = env_int("SPMV_B200_PR_SMALL", 1);
    static const int max_rows = env_int("SPMV_B200_PR_SMALL_ROWS", 8192);
    static const int max_nnz = env_int("SPMV_B200_PR_SMALL_NNZ", 1 << 18);
    if (mode == 0 || n <= 0) return false;
    return mode == 2 || (n <= max_rows && nnz <= max_nnz);
}

// Runs the loop.  r0 = buf_a holds 1/n, d_dsum its dangling mass, d_bits the dangling bitmask (set up by the caller
// exactly as for the multi-kernel loop), d_pvec the personalization vector or nullptr.  *final_buffer: 0 = buf_a,
// 1 = buf_b.  cudaErrorNotSupported: the device cannot launch cooperatively -- the caller takes the multi-kernel loop.
cudaError_t pagerank_small_run(const CsrView& A, float damping, float tolerance, int max_iterations, const uint32_t* d_bits,
                               float* buf_a, float* buf_b, const float* d_dsum, float* l2_history, int history_capacity,
                               int* iterations, float* residual, double* l1, bool* converged, int* final_buffer,
                               cudaStream_t stream, const float* d_pvec) {
    int dev = 0, coop = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (!coop || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pagerank_small_kernel, kSmallThreads, 0) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        return cudaErrorNotSupported;
    }
    int blocks = (A.rows + kSmallWarps - 1) / kSmallWarps;
    if (blocks > sms) blocks = sms;
    if (blocks < 1) blocks = 1;
    const int hist = (l2_history && history_capacity > 0) ? (history_capacity < max_iterations ? history_capacity : max_iterations) : 0;
    // one device block: partials | barrier | outputs | history
    const size_t partial_bytes = sizeof(double) * 2 * blocks * 3;
    const size_t bytes = partial_bytes + 64 + 64 + sizeof(float) * static_cast<size_t>(hist > 0 ? hist : 1);
    unsigned char* block = nullptr;
    cudaError_t e = cudaMalloc(&block, bytes);
    if (e != cudaSuccess) return e;
    cudaMemsetAsync(block, 0, bytes, stream);
    SmallArgs a;
    a.A = A;
    a.damping = damping;
    a.teleport = d_pvec ? 1.0f - damping : (1.0f - damping) / A.rows;  // reference src/pagerank.cu:86
    a.pvec = d_pvec;
    a.tolerance = tolerance;
    a.max_iterations = max_iterations;
    a.bits = d_bits;
    a.buf[0] = buf_a;
    a.buf[1] = buf_b;
    a.dsum0 = d_dsum;
    a.partials = reinterpret_cast<double*>(block);
    a.barrier = reinterpret_cast<unsigned*>(block + partial_bytes);
    a.out_l1 = reinterpret_cast<double*>(block + partial_bytes + 64);
    a.out_residual = reinterpret_cast<float*>(block + partial_bytes + 64 + 8);
    a.out_i = reinterpret_cast<int*>(block + partial_bytes + 64 + 16);
    a.history = hist > 0 ? reinterpret_cast<float*>(block + partial_bytes + 128) : nullptr;
    a.history_capacity = hist;
    void* params[] = {&a};
    e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(pagerank_small_kernel), dim3(blocks), dim3(kSmallThreads), params, 0, stream);
    count_launches(1);
    struct { double l1; float residual; float pad; int i[3]; } out;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&out, block + partial_bytes + 64, sizeof(out), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e == cudaSuccess) {
        if (iterations) *iterations = out.i[0];
        if (converged) *converged = out.i[1] != 0;
        if (final_buffer) *final_buffer = out.i[2];
        if (residual) *residual = out.residual;
        if (l1) *l1 = out.l1;
        if (hist > 0 && out.i[0] > 0)
            e = cudaMemcpy(l2_history, a.history, sizeof(float) * static_cast<size_t>(out.i[0] < hist ? out.i[0] : hist), cudaMemcpyDeviceToHost);
    }
    cudaFree(block);
    return e;
}

}  // namespace b200
}  // namespace spmv
