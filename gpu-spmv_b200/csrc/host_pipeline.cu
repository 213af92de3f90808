// host_pipeline.cu -- y_host = A * x_host for an ELL matrix that is resident in HBM while the
// vectors live in HOST memory: the end-to-end form of the hot path (what a caller of the reference
// does around spmv_ell: cudaMemcpy x up, spmv_ell, cudaMemcpy y down -- reference README.md:98-118,
// src/benchmark.cu:36-38,95-102).  Done serially that is H2D + kernel + D2H; the kernel is 5 % of it.
//
// Here the three legs are pipelined over row chunks on three streams:
//     copy stream    x chunk 0, 1, 2, ...                      (H2D, PCIe down-link)
//     compute stream rows of chunk c as soon as the x entries THEY read have arrived
//     drain stream   y chunk c as soon as chunk c is computed  (D2H, PCIe up-link)
// Which x entries a row chunk reads is a property of the matrix, measured once per plan on the
// device: the column range [min col, max col] of every row chunk.  A banded matrix (BASELINE
// config 2: the 5-point Laplacian reads x[i - 4096 .. i + 4096]) then overlaps the up- and
// down-link almost completely (PCIe is full duplex); a matrix whose rows read all of x
// degenerates to H2D, then compute overlapped with D2H -- never worse than the serial form.
// Numerics: the row chunks run the same ELL kernel (ell_tma_pipe_kernel<1>) on the same rows, so
// y is bit-identical to spmv_ell / spmv_cpu_ell.
//
// Default form (the "chunked" form above stays as SPMV_B200_HOST_GATED=0 and as the fall-back): the
// GATED form of ell_gated_kernel.cu -- ONE upload copy, ONE persistent kernel that consumes x while it
// arrives (the data is its own arrival flag), and one stream-ordered wait + D2H copy per row chunk
// queued before the launch, released by progress counters the kernel advances.  Measurements:
// profiles/r2_host_gated.txt.
#include "internal.hpp"

#include <cuda.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <vector>

namespace spmv {
namespace b200 {

cudaError_t launch_ell_rows(int rows, int width, const int* col_indices, const float* values, const float* x, float* y,
                            int row_lo, int row_hi, cudaStream_t stream);
// ell_gated_kernel.cu
bool ell_gated_applies(int rows, int width, const int* col_indices, const float* values);
int ell_gated_windows(int rows);
int ell_gated_window_rows();
int ell_gated_warps_per_window();
cudaError_t launch_ell_window_max_col(int rows, int width, const int* col_indices, int* d_wmax, cudaStream_t stream);
cudaError_t launch_fill_sentinel(float* x, size_t n, cudaStream_t stream);
cudaError_t launch_ell_gated(int rows, int width, const int* col_indices, const float* values, const float* x, float* y,
                             const int* d_window_poll, const unsigned* d_done_flag, unsigned epoch, unsigned* abort_word,
                             unsigned* abort_host, unsigned long long timeout_ns, unsigned poll_sleep_ns, unsigned* d_progress,
                             const unsigned char* d_window_chunk, const unsigned* d_chunk_warps, unsigned* ready_host,
                             cudaStream_t stream);

namespace {

// min / max column (padding excluded) of every row chunk; chunk c = rows [c * chunk_rows, ...).  A block owns a
// contiguous run of rows (32-bit indexing, coalesced slices), reduces per chunk it touches and issues one atomic pair.
__global__ void ell_chunk_col_range_kernel(int rows, int width, const int* __restrict__ col_indices, int chunk_rows,
                                           int* __restrict__ cmin, int* __restrict__ cmax) {
    const int per_block = (rows + gridDim.x - 1) / gridDim.x;
    const int r_begin = min(rows, static_cast<int>(blockIdx.x) * per_block), r_end = min(rows, r_begin + per_block);
    __shared__ int s_lo[8], s_hi[8];
    for (int c = r_begin / chunk_rows; c * static_cast<long long>(chunk_rows) < r_end; ++c) {  // the chunks this block touches
        const int lo_row = max(r_begin, c * chunk_rows), hi_row = static_cast<int>(min(static_cast<long long>(r_end), (c + 1LL) * chunk_rows));
        int lo = INT_MAX, hi = -1;
        for (int row = lo_row + threadIdx.x; row < hi_row; row += blockDim.x)
            for (int k = 0; k < width; ++k) {
                const int v = col_indices[static_cast<size_t>(k) * rows + row];
                if (v >= 0) { lo = min(lo, v); hi = max(hi, v); }
            }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if ((threadIdx.x & 31) == 0) { s_lo[threadIdx.x >> 5] = lo; s_hi[threadIdx.x >> 5] = hi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < static_cast<int>(blockDim.x >> 5); ++w) { lo = min(lo, s_lo[w]); hi = max(hi, s_hi[w]); }
            if (hi >= 0) { atomicMin(cmin + c, lo); atomicMax(cmax + c, hi); }
        }
        __syncthreads();
    }
}

// the device address of a page-locked, device-mapped host buffer (nullptr: y_host is something else, or
// SPMV_B200_HOST_ZERO_COPY_Y=0)
float* mapped_device_pointer(float* y_host) {
    static const int zero_copy = env_int("SPMV_B200_HOST_ZERO_COPY_Y", 1);
    if (!zero_copy) return nullptr;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, y_host) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
        return static_cast<float*>(attr.devicePointer);
    cudaGetLastError();
    return nullptr;
}

// cuStreamWriteValue32: a stream-ordered 32-bit store executed by the stream's front
// end (no SM, no copy descriptor) -- looked up at run time like every driver entry point of this library (symm.cpp)
using StreamValue32Fn = CUresult (*)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
StreamValue32Fn driver_entry(const char* name) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        p = nullptr;
    }
    return reinterpret_cast<StreamValue32Fn>(p);
}
StreamValue32Fn write_value32() {
    static const StreamValue32Fn fn = driver_entry("cuStreamWriteValue32");
    return fn;
}
}  // namespace

struct EllHostPlan {
    int rows = 0, cols = 0, width = 0;
    const int* d_cols = nullptr;      // the matrix (borrowed: must outlive the plan)
    const float* d_vals = nullptr;
    int chunks = 0, chunk_rows = 0;   // row chunks
    int x_chunks = 0, x_chunk = 0;    // x chunks (entries)
    std::vector<int> need;            // last x chunk a row chunk reads (-1: none)
    std::vector<char> x_needed;       // x chunks some row reads: the others are never uploaded (a row shard of a
                                      // larger system reads only its own band of x)
    bool ranged = false;              // the row-range kernel applies; else one launch after all of x
    float* d_x = nullptr;
    float* d_y = nullptr;
    cudaStream_t s_up = nullptr, s_run = nullptr, s_down = nullptr;
    std::vector<cudaEvent_t> ev_x, ev_y;
    cudaEvent_t ev_start = nullptr;
    // gated form
    bool gated = false;
    int g_chunks = 0;                 // row chunks of the download
    std::vector<int> g_first;         // [g_chunks + 1] first 256-row window of every chunk
    unsigned char* d_window_chunk = nullptr;  // per window: its chunk
    unsigned* d_chunk_warps = nullptr;        // per chunk: consumer warps that report
    size_t up_lo = 0, up_hi = 0;      // x entries [up_lo, up_hi) travel (what some row reads, at x_chunk granularity)
    int* d_poll = nullptr;            // per window: the largest column it reads
    unsigned* d_done = nullptr;       // epoch of the call whose upload is complete
    unsigned* d_progress = nullptr;   // [g_chunks] consumer warps done in the current call
    unsigned* h_ready = nullptr;      // [g_chunks] epoch of the call whose chunk is complete (mapped, page-locked: the kernel writes it)
    unsigned* h_ready_dev = nullptr;  // its device address
    unsigned* d_abort = nullptr;      // device word: a producer timed out
    unsigned* h_abort = nullptr;      // the same for the host (mapped, page-locked)
    unsigned* h_abort_dev = nullptr;  // its device address
    unsigned epoch = 0;
    cudaStream_t s_down2 = nullptr;
    cudaEvent_t ev_up = nullptr, ev_fill = nullptr, ev_kernel = nullptr;
    ~EllHostPlan() {
        if (s_run) cudaStreamSynchronize(s_run);  // the sentinel refill of the last call may still be running
        cudaFree(d_poll); cudaFree(d_done); cudaFree(d_progress); cudaFree(d_abort); cudaFree(d_window_chunk); cudaFree(d_chunk_warps);
        if (h_abort) cudaFreeHost(h_abort);
        if (h_ready) cudaFreeHost(h_ready);
        if (s_down2) cudaStreamDestroy(s_down2);
        if (ev_up) cudaEventDestroy(ev_up);
        if (ev_fill) cudaEventDestroy(ev_fill);
        if (ev_kernel) cudaEventDestroy(ev_kernel);
        for (auto e : ev_x) cudaEventDestroy(e);
        for (auto e : ev_y) cudaEventDestroy(e);
        if (ev_start) cudaEventDestroy(ev_start);
        if (s_up) cudaStreamDestroy(s_up);
        if (s_run) cudaStreamDestroy(s_run);
        if (s_down) cudaStreamDestroy(s_down);
        cudaFree(d_x);
        cudaFree(d_y);
    }
};

int ell_host_plan_create(const ELLMatrix* A, int chunks, EllHostPlan** out) {
    if (!A || !out) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (!A->d_col_indices || !A->d_values) return static_cast<int>(SpMVError::INVALID_FORMAT);
    EllHostPlan* p = new (std::nothrow) EllHostPlan();
    if (!p) return static_cast<int>(SpMVError::OUT_OF_MEMORY);
    p->rows = A->num_rows; p->cols = A->num_cols; p->width = A->max_nnz_per_row;
    p->d_cols = A->d_col_indices; p->d_vals = A->d_values;
    if (chunks <= 0) chunks = 12;  // measured on B200 / PCIe Gen5 (config 2, y stored straight into pinned memory): 6 / 8 / 12 / 16 / 24 / 32 chunks -> 1.85 / 1.78 / 1.72 / 1.78 / 1.82 / 1.81 ms (through a staging buffer + cudaMemcpyAsync per chunk: 1.88 / 1.84 / 1.83 / 1.88 / 2.03 / 2.18 ms)
    // chunk boundaries on multiples of 1024 rows / entries: TMA slices and copies stay 16-byte aligned
    auto round_up = [](long long v, long long m) { return (v + m - 1) / m * m; };
    p->chunk_rows = static_cast<int>(std::max<long long>(1024, round_up((static_cast<long long>(p->rows) + chunks - 1) / chunks, 1024)));
    p->chunks = p->rows > 0 ? (p->rows + p->chunk_rows - 1) / p->chunk_rows : 0;
    // x travels in chunks of the same size as the rows.  (Measured: finer x chunks -- 4 or 8 per row chunk, so that
    // a banded row chunk waits for less beyond its own rows -- cost more in per-copy overhead than they gain:
    // 2.09 / 2.31 ms against 1.83 ms; SPMV_B200_HOST_X_SPLIT keeps the experiment reproducible.)
    static const int x_per_row_chunk = std::min(16, std::max(1, env_int("SPMV_B200_HOST_X_SPLIT", 1)));
    const long long xc = static_cast<long long>(chunks) * x_per_row_chunk;
    p->x_chunk = static_cast<int>(std::max<long long>(1024, round_up((static_cast<long long>(p->cols) + xc - 1) / xc, 1024)));
    p->x_chunks = p->cols > 0 ? (p->cols + p->x_chunk - 1) / p->x_chunk : 0;
    bool ok = cudaMalloc(&p->d_x, sizeof(float) * static_cast<size_t>(std::max(p->cols, 1))) == cudaSuccess &&
              cudaMalloc(&p->d_y, sizeof(float) * static_cast<size_t>(std::max(p->rows, 1))) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->s_up, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->s_run, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->s_down, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&p->ev_start, cudaEventDisableTiming) == cudaSuccess;
    p->ev_x.assign(p->x_chunks, nullptr);
    p->ev_y.assign(p->chunks, nullptr);
    for (auto& e : p->ev_x) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    for (auto& e : p->ev_y) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    p->need.assign(p->chunks, p->x_chunks - 1);
    p->x_needed.assign(p->x_chunks, 1);
    // does the row-range kernel apply to this matrix?  (same test as launch_ell_rows)
    p->ranged = p->width >= 1 && p->width <= 8 && p->rows % 4 == 0 &&
                ((reinterpret_cast<uintptr_t>(p->d_cols) | reinterpret_cast<uintptr_t>(p->d_vals)) & 15u) == 0;
    if (ok && p->ranged && p->chunks > 0 && p->width > 0) {
        int *d_min = nullptr, *d_max = nullptr;
        std::vector<int> h_min(p->chunks, INT_MAX), h_max(p->chunks, -1);
        ok = cudaMalloc(&d_min, sizeof(int) * p->chunks) == cudaSuccess && cudaMalloc(&d_max, sizeof(int) * p->chunks) == cudaSuccess;
        if (ok) {
            cudaMemcpy(d_min, h_min.data(), sizeof(int) * p->chunks, cudaMemcpyHostToDevice);
            cudaMemcpy(d_max, h_max.data(), sizeof(int) * p->chunks, cudaMemcpyHostToDevice);
            ell_chunk_col_range_kernel<<<148 * 8, 256>>>(p->rows, p->width, p->d_cols, p->chunk_rows, d_min, d_max);
            count_launches(1);
            ok = cudaMemcpy(h_min.data(), d_min, sizeof(int) * p->chunks, cudaMemcpyDeviceToHost) == cudaSuccess &&
                 cudaMemcpy(h_max.data(), d_max, sizeof(int) * p->chunks, cudaMemcpyDeviceToHost) == cudaSuccess;
            // x chunks are uploaded in index order on one stream, so "the last chunk read" is what a row chunk waits for
            for (int c = 0; ok && c < p->chunks; ++c) p->need[c] = h_max[c] < 0 ? -1 : std::min(h_max[c], p->cols - 1) / p->x_chunk;
            if (ok) {
                p->x_needed.assign(p->x_chunks, 0);
                for (int c = 0; c < p->chunks; ++c) {
                    if (h_max[c] < 0) continue;
                    const int lo = std::max(h_min[c], 0) / p->x_chunk, hi = p->need[c];
                    for (int j = lo; j <= hi; ++j) p->x_needed[j] = 1;
                }
            }
        }
        cudaFree(d_min);
        cudaFree(d_max);
    }
    // gated form: per-window poll table, completion flag, progress counters, abort words, second download stream
    if (ok && p->ranged && env_int("SPMV_B200_HOST_GATED", 1) && write_value32() &&
        ell_gated_applies(p->rows, p->width, p->d_cols, p->d_vals)) {
        const int windows = ell_gated_windows(p->rows);
        // Download chunks: equal ones.  Every D2H copy costs ~19 us of idle down-link on B200 (its completion is a PCIe
        // round trip under load) and the download trails the product by one chunk: 6 / 8 / 10 / 12 chunks -> 1.663 /
        // 1.640 / 1.669 / 1.683 ms on config 2; a small first chunk followed by growing ones (the download is the
        // slower direction) was measured too and loses to 8 equal chunks (1.71-1.96 ms) -- profiles/r2_host_gated.txt
        {
            const int want = std::min(255, std::max(1, env_int("SPMV_B200_HOST_GATED_CHUNKS", 8)));
            const int size = (windows + want - 1) / want;
            p->g_first.assign(1, 0);
            while (p->g_first.back() < windows) p->g_first.push_back(std::min(windows, p->g_first.back() + size));
            p->g_chunks = static_cast<int>(p->g_first.size()) - 1;
        }
        int first = 0, last = p->x_chunks - 1;
        while (first < p->x_chunks && !p->x_needed[first]) ++first;
        while (last >= first && !p->x_needed[last]) --last;
        p->up_lo = static_cast<size_t>(first) * p->x_chunk;
        p->up_hi = last < first ? p->up_lo : std::min<size_t>(static_cast<size_t>(p->cols), static_cast<size_t>(last + 1) * p->x_chunk);
        bool g = cudaMalloc(&p->d_poll, sizeof(int) * windows) == cudaSuccess &&
                 cudaMalloc(&p->d_done, sizeof(unsigned)) == cudaSuccess &&
                 cudaMalloc(&p->d_progress, sizeof(unsigned) * p->g_chunks) == cudaSuccess &&
                 cudaMalloc(&p->d_window_chunk, windows) == cudaSuccess &&
                 cudaMalloc(&p->d_chunk_warps, sizeof(unsigned) * p->g_chunks) == cudaSuccess &&
                 cudaMalloc(&p->d_abort, sizeof(unsigned)) == cudaSuccess &&
                 cudaHostAlloc(&p->h_abort, sizeof(unsigned), cudaHostAllocMapped) == cudaSuccess &&
                 cudaHostGetDevicePointer(&p->h_abort_dev, p->h_abort, 0) == cudaSuccess &&
                 cudaHostAlloc(&p->h_ready, sizeof(unsigned) * p->g_chunks, cudaHostAllocMapped) == cudaSuccess &&
                 cudaHostGetDevicePointer(&p->h_ready_dev, p->h_ready, 0) == cudaSuccess &&
                 cudaStreamCreateWithFlags(&p->s_down2, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&p->ev_up, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&p->ev_fill, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&p->ev_kernel, cudaEventDisableTiming) == cudaSuccess &&
                 cudaMemset(p->d_done, 0, sizeof(unsigned)) == cudaSuccess &&
                 cudaMemset(p->d_progress, 0, sizeof(unsigned) * p->g_chunks) == cudaSuccess &&
                 cudaMemset(p->d_abort, 0, sizeof(unsigned)) == cudaSuccess &&
                 launch_ell_window_max_col(p->rows, p->width, p->d_cols, p->d_poll, nullptr) == cudaSuccess &&
                 launch_fill_sentinel(p->d_x, static_cast<size_t>(std::max(p->cols, 1)), nullptr) == cudaSuccess &&
                 cudaEventRecord(p->ev_fill, nullptr) == cudaSuccess &&
                 cudaDeviceSynchronize() == cudaSuccess;
        if (g) {
            std::vector<unsigned char> wc(windows);
            std::vector<unsigned> cw(p->g_chunks);
            for (int c = 0; c < p->g_chunks; ++c) {
                cw[c] = static_cast<unsigned>(p->g_first[c + 1] - p->g_first[c]) * static_cast<unsigned>(ell_gated_warps_per_window());
                for (int w = p->g_first[c]; w < p->g_first[c + 1]; ++w) wc[w] = static_cast<unsigned char>(c);
            }
            g = cudaMemcpy(p->d_window_chunk, wc.data(), windows, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemcpy(p->d_chunk_warps, cw.data(), sizeof(unsigned) * p->g_chunks, cudaMemcpyHostToDevice) == cudaSuccess;
        }
        if (g) {
            *p->h_abort = 0;
            for (int c = 0; c < p->g_chunks; ++c) p->h_ready[c] = 0;
        } else {
            cudaGetLastError();
        }
        p->gated = g;
    }
    if (!ok) {
        cudaGetLastError();
        delete p;
        return static_cast<int>(SpMVError::CUDA_MALLOC);
    }
    *out = p;
    return 0;
}

void ell_host_plan_destroy(EllHostPlan* p) { delete p; }

namespace {

// The gated form.  0: y is complete; 1: the kernel gave up waiting (nothing usable in y: the caller runs the
// chunked form and stops using this one); < 0: CUDA error.
int run_gated(EllHostPlan* p, const float* x_host, float* y_host) {
    static const int down_streams = std::min(2, std::max(1, env_int("SPMV_B200_HOST_DOWN_STREAMS", 1)));
    static const unsigned long long timeout_ns = 1000000ull * static_cast<unsigned long long>(std::max(1, env_int("SPMV_B200_HOST_GATED_TIMEOUT_MS", 2000)));
    static const unsigned poll_sleep_ns = static_cast<unsigned>(std::max(0, env_int("SPMV_B200_HOST_GATED_POLL_NS", 200)));
    static const bool trace = getenv("SPMV_B200_TRACE") != nullptr;
    const StreamValue32Fn write32 = write_value32();
    const unsigned epoch = ++p->epoch == 0 ? ++p->epoch : p->epoch;  // flags start at 0: never a valid epoch
    cudaStream_t downs[2] = {p->s_down, down_streams > 1 ? p->s_down2 : p->s_down};
    const int rows_per_window = ell_gated_window_rows();
    const int windows = ell_gated_windows(p->rows);
    const auto t_begin = std::chrono::steady_clock::now();
    auto since_begin_us = [&] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_begin).count(); };
    bool ok = true;
    // order after whatever the caller queued on the legacy stream (matrix upload, ...)
    ok = ok && cudaEventRecord(p->ev_start, nullptr) == cudaSuccess;
    for (cudaStream_t s : {p->s_up, p->s_run, p->s_down, p->s_down2}) ok = ok && cudaStreamWaitEvent(s, p->ev_start, 0) == cudaSuccess;
    // up: one copy over the sentinels (which the previous call re-laid after its product), then the completion flag
    ok = ok && cudaStreamWaitEvent(p->s_up, p->ev_fill, 0) == cudaSuccess;
    // SPMV_B200_HOST_GATED_TEST_STALL=1 (tests only): the upload never happens, so the kernel must time out, drain and hand the
    // call to the chunked form -- the path that guarantees the call cannot hang
    static const int test_stall = env_int("SPMV_B200_HOST_GATED_TEST_STALL", 0);
    if (ok && p->up_hi > p->up_lo && !test_stall)
        ok = cudaMemcpyAsync(p->d_x + p->up_lo, x_host + p->up_lo, (p->up_hi - p->up_lo) * sizeof(float), cudaMemcpyHostToDevice, p->s_up) == cudaSuccess;
    if (!test_stall) ok = ok && write32(reinterpret_cast<CUstream>(p->s_up), reinterpret_cast<CUdeviceptr>(p->d_done), epoch, 0) == CUDA_SUCCESS;
    ok = ok && cudaEventRecord(p->ev_up, p->s_up) == cudaSuccess;
    if (!ok) return -1;
    // the product, consuming x as it lands; then (once the upload is over, too) the sentinels for the next call
    // y in page-locked, device-mapped host memory (cudaHostAlloc / cudaHostRegister: what a pinned buffer is under UVA):
    // the kernel stores its rows STRAIGHT into y_host -- 128-byte posted PCIe writes that leave as the rows are
    // finished, in step with the upload: 1.47 ms on config 2 against 1.64 ms with 8 D2H copies (each copy costs ~19 us
    // of idle link), profiles/r2_host_gated.txt.  Any other y_host goes down in D2H chunks.
    float* y_direct = mapped_device_pointer(y_host);
    ok = (y_direct || cudaMemsetAsync(p->d_progress, 0, sizeof(unsigned) * p->g_chunks, p->s_run) == cudaSuccess) &&
         launch_ell_gated(p->rows, p->width, p->d_cols, p->d_vals, p->d_x, y_direct ? y_direct : p->d_y, p->d_poll, p->d_done, epoch, p->d_abort,
                          p->h_abort_dev, timeout_ns, poll_sleep_ns, y_direct ? nullptr : p->d_progress, p->d_window_chunk, p->d_chunk_warps,
                          p->h_ready_dev, p->s_run) == cudaSuccess &&
         cudaEventRecord(p->ev_kernel, p->s_run) == cudaSuccess;
    const bool launched = ok;
    ok = ok && cudaStreamWaitEvent(p->s_run, p->ev_up, 0) == cudaSuccess;
    ok = ok && launch_fill_sentinel(p->d_x + p->up_lo, p->up_hi - p->up_lo, p->s_run) == cudaSuccess;
    ok = ok && cudaEventRecord(p->ev_fill, p->s_run) == cudaSuccess;
    const double t_queued = since_begin_us();
    // down: this thread watches the ready words the kernel writes and queues the copy of a chunk the moment it is complete
    std::vector<double> t_ready(trace ? p->g_chunks : 0);
    for (int c = 0; launched && ok && !y_direct && c < p->g_chunks; ++c) {
        volatile unsigned* ready = p->h_ready + c;
        unsigned spins = 0;
        while (*ready != epoch) {
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
            if ((++spins & 0x3fffu) == 0) {  // a failed kernel must not leave this thread spinning
                const cudaError_t q = cudaStreamQuery(p->s_run);
                if ((q != cudaSuccess && q != cudaErrorNotReady) || since_begin_us() > 30e6) { ok = false; break; }
                if (q == cudaSuccess && *ready != epoch) { ok = false; break; }
            }
        }
        if (!ok) break;
        if (trace) t_ready[c] = since_begin_us();
        const int w_lo = p->g_first[c], w_hi = p->g_first[c + 1];
        const size_t lo = static_cast<size_t>(w_lo) * rows_per_window;
        const size_t hi = std::min<size_t>(static_cast<size_t>(p->rows), static_cast<size_t>(w_hi) * rows_per_window);
        ok = cudaMemcpyAsync(y_host + lo, p->d_y + lo, (hi - lo) * sizeof(float), cudaMemcpyDeviceToHost, downs[c & 1]) == cudaSuccess;
    }
    if (y_direct && launched) ok = cudaEventSynchronize(p->ev_kernel) == cudaSuccess && ok;  // the kernel's own stores are the download
    ok = cudaStreamSynchronize(p->s_down) == cudaSuccess && ok;
    ok = cudaStreamSynchronize(p->s_down2) == cudaSuccess && ok;
    ok = cudaStreamSynchronize(p->s_up) == cudaSuccess && ok;
    if (trace) {
        fprintf(stderr, "[gated] queued %.0f us; chunk ready at [us]:", t_queued);
        for (double t : t_ready) fprintf(stderr, " %.0f", t);
        fprintf(stderr, "; done %.0f us\n", since_begin_us());
    }
    if (!ok) return -1;
    if (*static_cast<volatile unsigned*>(p->h_abort) != 0) {
        cudaStreamSynchronize(p->s_run);
        *p->h_abort = 0;
        cudaMemset(p->d_abort, 0, sizeof(unsigned));
        return 1;
    }
    return 0;
}

}  // namespace

// Blocking: returns when y_host is complete.  x_host / y_host should be page-locked (cudaHostAlloc /
// cudaHostRegister) for the copies to overlap; pageable memory works but serialises.
int spmv_ell_host(EllHostPlan* p, const float* x_host, float* y_host) {
    NvtxRange nvtx_range("spmv_b200:spmv_ell_host");
    if (!p || !x_host || !y_host) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (p->rows <= 0) return 0;
    bool ok = true;
    if (p->gated) {
        const int rc = run_gated(p, x_host, y_host);
        if (rc == 0) return 0;
        cudaGetLastError();
        for (cudaStream_t s : {p->s_up, p->s_run, p->s_down, p->s_down2}) cudaStreamSynchronize(s);
        cudaGetLastError();
        p->gated = false;  // the chunked form from now on
        if (rc < 0) return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    // order after whatever the caller queued on the legacy stream (matrix upload, ...)
    ok = ok && cudaEventRecord(p->ev_start, nullptr) == cudaSuccess;
    ok = ok && cudaStreamWaitEvent(p->s_up, p->ev_start, 0) == cudaSuccess;
    ok = ok && cudaStreamWaitEvent(p->s_run, p->ev_start, 0) == cudaSuccess;
    for (int j = 0; ok && j < p->x_chunks; ++j) {
        if (!p->x_needed[j]) continue;
        const size_t lo = static_cast<size_t>(j) * p->x_chunk;
        const size_t n = std::min<size_t>(p->x_chunk, static_cast<size_t>(p->cols) - lo);
        ok = cudaMemcpyAsync(p->d_x + lo, x_host + lo, n * sizeof(float), cudaMemcpyHostToDevice, p->s_up) == cudaSuccess &&
             cudaEventRecord(p->ev_x[j], p->s_up) == cudaSuccess;
    }
    if (ok && !p->ranged) {  // one launch over the whole matrix once all of x is there
        if (p->x_chunks > 0) ok = cudaStreamWaitEvent(p->s_run, p->ev_x[p->x_chunks - 1], 0) == cudaSuccess;
        ok = ok && launch_ell(p->rows, p->width, p->d_cols, p->d_vals, p->d_x, p->d_y, nullptr, p->s_run) == cudaSuccess;
        ok = ok && cudaMemcpyAsync(y_host, p->d_y, sizeof(float) * static_cast<size_t>(p->rows), cudaMemcpyDeviceToHost, p->s_run) == cudaSuccess;
        ok = ok && cudaStreamSynchronize(p->s_run) == cudaSuccess;
    } else if (ok) {
        // y in page-locked, device-mapped host memory (cudaHostAlloc / cudaHostRegister: what a pinned buffer is
        // under UVA): the kernel stores its rows STRAIGHT into y_host over PCIe -- the download is the kernel's
        // own posted writes, overlapped row by row with the product, no staging buffer, no per-chunk copy.
        float* y_direct = mapped_device_pointer(y_host);
        int waited = -1;  // highest x chunk the compute stream already waits for
        for (int c = 0; ok && c < p->chunks; ++c) {
            const int lo = c * p->chunk_rows, hi = std::min(p->rows, lo + p->chunk_rows);
            if (p->need[c] > waited) {
                ok = cudaStreamWaitEvent(p->s_run, p->ev_x[p->need[c]], 0) == cudaSuccess;
                waited = p->need[c];
            }
            ok = ok && launch_ell_rows(p->rows, p->width, p->d_cols, p->d_vals, p->d_x, y_direct ? y_direct : p->d_y, lo, hi, p->s_run) == cudaSuccess;
            if (y_direct) continue;
            ok = ok && cudaEventRecord(p->ev_y[c], p->s_run) == cudaSuccess;
            ok = ok && cudaStreamWaitEvent(p->s_down, p->ev_y[c], 0) == cudaSuccess;
            ok = ok && cudaMemcpyAsync(y_host + lo, p->d_y + lo, sizeof(float) * static_cast<size_t>(hi - lo),
                                       cudaMemcpyDeviceToHost, p->s_down) == cudaSuccess;
        }
        ok = ok && cudaStreamSynchronize(y_direct ? p->s_run : p->s_down) == cudaSuccess;
        ok = cudaStreamSynchronize(p->s_up) == cudaSuccess && ok;  // x chunks no row read (none for a square matrix)
    }
    if (!ok) {
        cudaGetLastError();
        cudaStreamSynchronize(p->s_up); cudaStreamSynchronize(p->s_run); cudaStreamSynchronize(p->s_down);
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

// bytes one call moves over PCIe: the x chunks some row reads, and y
void ell_host_plan_bytes(const EllHostPlan* p, unsigned long long* h2d, unsigned long long* d2h) {
    unsigned long long up = 0;
    if (p && p->gated) {
        up = sizeof(float) * static_cast<unsigned long long>(p->up_hi - p->up_lo);
    } else if (p) {
        for (int j = 0; j < p->x_chunks; ++j) {
            if (!p->x_needed[j]) continue;
            const size_t lo = static_cast<size_t>(j) * p->x_chunk;
            up += sizeof(float) * std::min<size_t>(p->x_chunk, static_cast<size_t>(p->cols) - lo);
        }
    }
    if (h2d) *h2d = up;
    if (d2h) *d2h = p ? sizeof(float) * static_cast<unsigned long long>(p->rows) : 0;
}

// whether the next call takes the gated form, and how many row chunks its download uses
void ell_host_plan_gated(const EllHostPlan* p, int* gated, int* down_chunks) {
    if (gated) *gated = p && p->gated ? 1 : 0;
    if (down_chunks) *down_chunks = p && p->gated ? p->g_chunks : 0;
}

void ell_host_plan_info(const EllHostPlan* p, int* chunks, int* ranged, int* max_lookahead) {
    if (chunks) *chunks = p ? p->chunks : 0;
    if (ranged) *ranged = p && p->ranged ? 1 : 0;
    if (max_lookahead) {  // how many x chunks beyond its own index a row chunk waits for, at most
        int m = 0;
        if (p) for (int c = 0; c < p->chunks; ++c) m = std::max(m, p->need[c] - c);
        *max_lookahead = m;
    }
}

}  // namespace b200
}  // namespace spmv
