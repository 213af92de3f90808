// dispatch.cu -- the device entry points of the API: spmv_csr / spmv_ell
// (reference src/spmv_kernels.cu:215-326, :328-420), their stream-ordered
// twins, and the kernel dispatch they share with the benchmark harness and
// PageRank.
//
// Contract kept from the reference launchers: argument checks in the same
// order with the same codes (null -> INVALID_ARGUMENT, vec_size mismatch ->
// INVALID_DIMENSION, missing device arrays -> INVALID_FORMAT), config == NULL
// -> {SCALAR_CSR, 256, false}, unknown kernel_type -> scalar, launch failure
// -> KERNEL_LAUNCH, and on success elapsed_ms (CUDA events around every kernel
// the call launches, merge-path partition and fix-up included), gflops =
// 2*nnz/(ms*1e6), bandwidth from the compulsory-bytes model, y = d_y.
// Differences (DESIGN.md, "launcher"): events are created once per thread and
// reused; use_texture and block_size are accepted and ignored; a matrix with
// zero rows succeeds with no launch (the reference reports KERNEL_LAUNCH for
// its 0-block grid); spmv_ell counts true non-zeros on the device instead of
// re-walking the host arrays after every call.
#include "internal.hpp"

#include <nvtx3/nvToolsExt.h>

#include <atomic>
#include <cstdlib>
#include <mutex>
#include <new>
#include <unordered_map>

namespace spmv {
namespace b200 {

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }


// ---- launch accounting ----------------------------------------------------------
static std::atomic<unsigned long long> g_launches{0};
void count_launches(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---- scratch ----------------------------------------------------------------------
Scratch::~Scratch() { release(); }
void Scratch::release() {
    if (ptr_) cudaFree(ptr_);
    ptr_ = nullptr;
    cap_ = 0;
}
void* Scratch::reserve(size_t bytes) {
    if (bytes <= cap_) return ptr_;
    if (ptr_) cudaFree(ptr_);
    ptr_ = nullptr;
    cap_ = 0;
    const size_t want = bytes + bytes / 4;  // head-room so slightly larger inputs do not reallocate
    if (cudaMalloc(&ptr_, want) != cudaSuccess) {
        cudaGetLastError();
        ptr_ = nullptr;
        return nullptr;
    }
    cap_ = want;
    return ptr_;
}

cudaError_t dispatch_csr(const CsrView& A, const float* x, float* y, int kernel_type, Scratch& scratch,
                         cudaStream_t stream, const PlannedCsr* planned) {
    if (A.rows <= 0) return cudaSuccess;
    switch (kernel_type) {
        case SpMVConfig::MERGE_PATH: {
            if (A.nnz <= 0) return launch_csr_stream(A, x, y, 1, stream);  // writes zeros
            if (planned && planned->seg.valid() && planned->seg.nnz == A.nnz && planned->seg.rows == A.rows &&
                planned->seg.cols == A.cols)
                return launch_seg_spmv(A, planned->seg, x, y, stream);
            void* block = scratch.reserve(merge_plan_bytes(A.rows, A.nnz, false));
            if (!block) return cudaErrorMemoryAllocation;
            const bool hub = planned && planned->hot.n_hot > 0 && planned->hot.nnz == A.nnz && planned->hot.cols == A.cols;
            // tile geometry by structure (7 or 8 items per thread): the same choice with and without a plan
            const MergePlan plan = merge_plan_carve(block, A.rows, A.nnz, false, merge_items_for(A.rows, A.nnz));
            cudaError_t e = launch_merge_partition(A, plan, stream);
            if (e != cudaSuccess) return e;
            if (hub) return launch_hot_spmv(A, planned->hot, x, y, plan, stream);
            return launch_merge_spmv(A, x, y, plan, stream);
        }
        case SpMVConfig::VECTOR_CSR:
            return launch_csr_vector(A, x, y, stream);
        case SpMVConfig::SCALAR_CSR:
        default:
            return launch_csr_stream(A, x, y, 1, stream);
    }
}

// ---- column plans ---------------------------------------------------------------------
// Explicit plan (additive API): merge coordinates computed once + the hub-column plan.
struct CsrPlan {
    CsrView A{};
    PlannedCsr planned;
    Scratch merge_block;
    MergePlan merge;
    // Opt-in (kPlanSnapshotValues): a uniform matrix is re-laid out as ELL on the device and
    // multiplied by the ELL kernel; ell_values is a SNAPSHOT of A.values (csr_plan_refresh_values).
    int ell_width = 0;
    float* ell_values = nullptr;
    int* ell_cols = nullptr;
};

constexpr int kPlanForce = 1;           // flags of csr_plan_create
constexpr int kPlanSnapshotValues = 2;
constexpr int kEllPlanMaxWidth = 8;     // the TMA-staged ELL pipeline (ell_kernels.cu) covers W <= 8

// ELL routing pays when the padding is small: rows * width <= 1.125 * nnz
static bool ell_route_worthwhile(const CsrView& A, int width) {
    return width >= 1 && width <= kEllPlanMaxWidth &&
           static_cast<long long>(A.rows) * width * 8 <= static_cast<long long>(A.nnz) * 9;
}

static cudaError_t longest_row(const CsrView& A, int* out, cudaStream_t stream) {
    int* d_w = nullptr;
    cudaError_t e = cudaMalloc(&d_w, sizeof(int));
    if (e != cudaSuccess) return e;
    cudaMemsetAsync(d_w, 0, sizeof(int), stream);
    e = launch_max_row_len(A, d_w, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_w, sizeof(int), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    cudaFree(d_w);
    return e;
}

// SPMV_B200_PLAN=hub|seg forces one of the planned kernels (tuning / tests); default: by structure
static int plan_kind_env() {
    static const int kind = [] {
        const char* v = getenv("SPMV_B200_PLAN");
        return !v ? 0 : (v[0] == 'h' ? 1 : (v[0] == 's' ? 2 : 0));
    }();
    return kind;
}

cudaError_t planned_build(const CsrView& A, PlannedCsr* out, int capacity, bool force, bool allow_seg,
                          cudaStream_t stream, bool prefer_seg) {
    out->release();
    if (A.rows <= 0 || A.nnz <= 0) return cudaSuccess;
    const int kind = plan_kind_env();
    if (kind == 2) return seg_plan_build(A, &out->seg, capacity, force, stream);
    const bool long_enough = static_cast<long long>(A.nnz) >= 4ll * A.rows;
    if (prefer_seg && kind == 0 && long_enough) {
        const cudaError_t e = seg_plan_build(A, &out->seg, capacity, force, stream);
        if (e != cudaSuccess || out->seg.valid()) return e;
    }
    // measured on R-MAT 24 / 26 and the Laplacian (profiles/r1_hub_kernel.md): the hub-column kernel wins
    // on scale-free matrices (and overlaps the PageRank slice exchange), the segmented stream elsewhere
    cudaError_t e = hot_plan_build(A, &out->hot, capacity, force, stream, 8);
    if (e != cudaSuccess || out->hot.n_hot > 0 || kind == 1 || !allow_seg) return e;
    if (!long_enough && !force) return cudaSuccess;
    return seg_plan_build(A, &out->seg, capacity, force, stream);
}

int csr_plan_create(const CSRMatrix* A, int max_hot_columns, int flags, CsrPlan** out) {
    NvtxRange nvtx_range("spmv_b200:csr_plan_create");
    const bool force = (flags & kPlanForce) != 0;
    if (!A || !out) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (!A->d_row_ptrs || !A->d_col_indices || (A->nnz > 0 && !A->d_values))
        return static_cast<int>(SpMVError::INVALID_FORMAT);
    CsrPlan* p = new (std::nothrow) CsrPlan();
    if (!p) return static_cast<int>(SpMVError::OUT_OF_MEMORY);
    p->A = view_of(A);
    cudaStream_t stream = nullptr;
    if (p->A.rows > 0 && p->A.nnz > 0) {
        void* block = p->merge_block.reserve(merge_plan_bytes(p->A.rows, p->A.nnz, false));
        if (!block) {
            delete p;
            return static_cast<int>(SpMVError::CUDA_MALLOC);
        }
        p->merge = merge_plan_carve(block, p->A.rows, p->A.nnz, false, merge_items_for(p->A.rows, p->A.nnz));
        cudaError_t e = cudaSuccess;
        if (flags & kPlanSnapshotValues) {  // uniform matrix -> ELL layout, if the caller accepts a value snapshot
            int width = 0;
            e = longest_row(p->A, &width, stream);
            if (e == cudaSuccess && ell_route_worthwhile(p->A, width)) {
                const size_t slots = static_cast<size_t>(p->A.rows) * width;
                if (cudaMalloc(&p->ell_values, slots * sizeof(float)) == cudaSuccess &&
                    cudaMalloc(&p->ell_cols, slots * sizeof(int)) == cudaSuccess) {
                    p->ell_width = width;
                    e = launch_ell_from_csr(p->A, width, p->ell_values, p->ell_cols, stream);
                } else {
                    cudaGetLastError();
                    cudaFree(p->ell_values);
                    p->ell_values = nullptr;
                }
            }
        }
        if (e == cudaSuccess) e = launch_merge_partition(p->A, p->merge, stream);
        if (e == cudaSuccess && p->ell_width == 0)
            e = planned_build(p->A, &p->planned, max_hot_columns, force, true, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p->planned.release();
            cudaFree(p->ell_values);
            cudaFree(p->ell_cols);
            delete p;
            return static_cast<int>(e == cudaErrorMemoryAllocation ? SpMVError::CUDA_MALLOC : SpMVError::KERNEL_LAUNCH);
        }
    }
    *out = p;
    return 0;
}

void csr_plan_destroy(CsrPlan* p) {
    if (!p) return;
    p->planned.release();
    cudaFree(p->ell_values);
    cudaFree(p->ell_cols);
    delete p;
}

void csr_plan_info(const CsrPlan* p, int* hot_columns, long long* hot_nnz, int* mode) {
    const bool seg = p && p->planned.seg.valid();
    if (hot_columns) *hot_columns = !p ? 0 : (seg ? p->planned.seg.n_hot : p->planned.hot.n_hot);
    if (hot_nnz) *hot_nnz = !p ? 0 : (seg ? p->planned.seg.hot_nnz : p->planned.hot.hot_nnz);
    if (mode) {
        if (p && p->ell_width > 0) *mode = 5;
        else if (seg) *mode = p->planned.seg.whole_x ? 4 : 3;
        else *mode = !p || p->planned.hot.n_hot <= 0 ? 0 : (p->planned.hot.all_hot ? 2 : 1);
    }
}

int spmv_csr_planned(const CsrPlan* p, const float* d_x, float* d_y, cudaStream_t stream) {
    NvtxRange nvtx_range("spmv_b200:spmv_csr_planned");
    if (!p || !d_x || !d_y) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    const CsrView& A = p->A;
    if (A.rows <= 0) return 0;
    cudaError_t e;
    if (A.nnz <= 0) e = launch_csr_stream(A, d_x, d_y, 1, stream);  // writes zeros
    else if (p->ell_width > 0) e = launch_ell(A.rows, p->ell_width, p->ell_cols, p->ell_values, d_x, d_y, nullptr, stream);
    else if (p->planned.seg.valid()) e = launch_seg_spmv(A, p->planned.seg, d_x, d_y, stream);
    else if (p->planned.hot.n_hot > 0) e = launch_hot_spmv(A, p->planned.hot, d_x, d_y, p->merge, stream);
    else e = launch_merge_spmv(A, d_x, d_y, p->merge, stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

// re-reads A.values into the ELL snapshot of a mode-5 plan (no-op for the other modes); stream-ordered
int csr_plan_refresh_values(CsrPlan* p, cudaStream_t stream) {
    if (!p) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (p->ell_width <= 0) return 0;
    if (launch_ell_from_csr(p->A, p->ell_width, p->ell_values, p->ell_cols, stream) != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

// Automatic plans for spmv_csr(MERGE_PATH) -- OPT-IN (spmv_b200_set_auto_plan(1) or
// SPMV_B200_AUTO_PLAN=1; off by default).  A plan holds a private re-encoding of col_indices and,
// for the segmented-stream kernel, of the row structure of row_ptrs; values and x are read live.
// The reference's struct fields are public, so a caller may legally rewrite d_col_indices /
// d_row_ptrs in place (or cudaFree them and get the same address back for another matrix of the
// same shape): with a plan attached that would silently multiply by the OLD sparsity pattern.  A
// drop-in must not change results by default, hence the opt-in; a caller that switches it on
// promises to call spmv_b200_csr_forget_plan after such an edit (INTEGRATION.md).  When on: only
// device arrays uploaded by csr_to_gpu / csr_from_coo_device are planned (the library sees them
// freed), on the second merge-path call over the same arrays; the plan costs 4 bytes per non-zero
// of device memory (+ 4 per non-empty row for the segmented stream).
namespace {
std::atomic<int> g_auto_plan_enabled{-1};  // -1: read SPMV_B200_AUTO_PLAN on first use

struct AutoEntry {
    int rows = 0, nnz = 0;
    int calls = 0;
    bool tried = false;
    PlannedCsr planned;
};
std::mutex g_auto_mu;
std::unordered_map<const void*, AutoEntry*> g_auto;
}  // namespace

int hot_env_mode() {
    static const int mode = env_int("SPMV_B200_HOT", -1);
    return mode;
}

bool auto_plan_enabled() {
    int v = g_auto_plan_enabled.load(std::memory_order_relaxed);
    if (v < 0) {
        v = env_int("SPMV_B200_AUTO_PLAN", 0) > 0 ? 1 : 0;
        g_auto_plan_enabled.store(v, std::memory_order_relaxed);
    }
    return v > 0;
}
void set_auto_plan(bool on) { g_auto_plan_enabled.store(on ? 1 : 0, std::memory_order_relaxed); }

void note_device_csr(const CSRMatrix* A) {
    if (!A || !A->d_col_indices || hot_env_mode() == 0) return;  // registered even while auto-plans are off: cheap, and the switch may come later
    std::lock_guard<std::mutex> lock(g_auto_mu);
    AutoEntry*& e = g_auto[A->d_col_indices];
    if (e) {
        e->planned.release();
        delete e;
    }
    e = new AutoEntry();
    e->rows = A->num_rows;
    e->nnz = A->nnz;
}

void forget_device_csr(const void* d_col_indices) {
    if (!d_col_indices) return;
    std::lock_guard<std::mutex> lock(g_auto_mu);
    auto it = g_auto.find(d_col_indices);
    if (it == g_auto.end()) return;
    it->second->planned.release();
    delete it->second;
    g_auto.erase(it);
}

// state of the automatic plan attached to A's device arrays (0 columns: none)
void auto_plan_info(const CSRMatrix* A, int* hot_columns, long long* hot_nnz) {
    if (hot_columns) *hot_columns = 0;
    if (hot_nnz) *hot_nnz = 0;
    if (!A || !A->d_col_indices) return;
    std::lock_guard<std::mutex> lock(g_auto_mu);
    auto it = g_auto.find(A->d_col_indices);
    if (it == g_auto.end()) return;
    const PlannedCsr& pl = it->second->planned;
    if (hot_columns) *hot_columns = pl.seg.valid() ? (pl.seg.n_hot > 0 ? pl.seg.n_hot : 1) : pl.hot.n_hot;
    if (hot_nnz) *hot_nnz = pl.seg.valid() ? pl.seg.hot_nnz : pl.hot.hot_nnz;
}

// nullptr: no plan (not an upload of ours, first call, or not worthwhile)
static const PlannedCsr* auto_planned(const CSRMatrix* A, cudaStream_t stream) {
    if (hot_env_mode() == 0 || !A->d_col_indices || !auto_plan_enabled()) return nullptr;
    std::lock_guard<std::mutex> lock(g_auto_mu);
    auto it = g_auto.find(A->d_col_indices);
    if (it == g_auto.end()) return nullptr;
    AutoEntry* e = it->second;
    if (e->rows != A->num_rows || e->nnz != A->nnz) return nullptr;  // the struct was edited by hand
    if (!e->tried && e->calls++ >= 1) {
        e->tried = true;
        if (planned_build(view_of(A), &e->planned, 0, hot_env_mode() > 0, true, stream) != cudaSuccess) {
            cudaGetLastError();
            e->planned.release();
        }
    }
    return e->planned.any() ? &e->planned : nullptr;
}

namespace {

// Per host thread and device: the two timing events, a merge-path scratch block
// and the 8-byte non-zero counter used by spmv_ell.
struct ThreadCtx {
    cudaEvent_t start = nullptr, stop = nullptr;
    Scratch scratch;
    unsigned long long* d_counter = nullptr;
    bool ok = false;
};

ThreadCtx* thread_ctx() {
    thread_local std::unordered_map<int, ThreadCtx*> per_device;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    auto it = per_device.find(dev);
    if (it != per_device.end()) return it->second->ok ? it->second : nullptr;
    ThreadCtx* c = new ThreadCtx();  // lives for the process (device resources outlive static dtors safely)
    c->ok = cudaEventCreate(&c->start) == cudaSuccess && cudaEventCreate(&c->stop) == cudaSuccess &&
            cudaMalloc(&c->d_counter, sizeof(unsigned long long)) == cudaSuccess;
    if (!c->ok) cudaGetLastError();
    per_device[dev] = c;
    return c->ok ? c : nullptr;
}

SpMVResult failed(SpMVError code) {
    SpMVResult r;
    r.error_code = static_cast<int>(code);
    return r;
}

// async stream scratch: one block per (device, stream), guarded by a mutex
std::mutex g_async_mu;
std::unordered_map<unsigned long long, Scratch*> g_async_scratch;

Scratch* async_scratch(cudaStream_t stream) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long key = (static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(stream)) << 6) ^
                                   static_cast<unsigned long long>(dev);
    std::lock_guard<std::mutex> lock(g_async_mu);
    auto it = g_async_scratch.find(key);
    if (it != g_async_scratch.end()) return it->second;
    Scratch* s = new Scratch();
    g_async_scratch[key] = s;
    return s;
}

}  // namespace

int spmv_csr_async(const CSRMatrix* A, const float* d_x, float* d_y, const SpMVConfig* config,
                   cudaStream_t stream) {
    if (!A || !d_x || !d_y) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (!A->d_row_ptrs || !A->d_col_indices || (A->nnz > 0 && !A->d_values))
        return static_cast<int>(SpMVError::INVALID_FORMAT);
    const int kernel = config ? static_cast<int>(config->kernel_type) : static_cast<int>(SpMVConfig::SCALAR_CSR);
    cudaError_t e = dispatch_csr(view_of(A), d_x, d_y, kernel, *async_scratch(stream), stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(e == cudaErrorMemoryAllocation ? SpMVError::CUDA_MALLOC : SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

int spmv_ell_async(const ELLMatrix* A, const float* d_x, float* d_y, cudaStream_t stream) {
    if (!A || !d_x || !d_y) return static_cast<int>(SpMVError::INVALID_ARGUMENT);
    if (!A->d_col_indices || !A->d_values) return static_cast<int>(SpMVError::INVALID_FORMAT);
    cudaError_t e = launch_ell(A->num_rows, A->max_nnz_per_row, A->d_col_indices, A->d_values, d_x, d_y, nullptr, stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return static_cast<int>(SpMVError::KERNEL_LAUNCH);
    }
    return 0;
}

}  // namespace b200

// ------------------------------------------------------------------- spmv_csr --
SpMVResult spmv_csr(const CSRMatrix* A, const float* d_x, float* d_y, const SpMVConfig* config, int vec_size) {
    b200::NvtxRange nvtx_range("spmv_b200:spmv_csr");
    if (!A || !d_x || !d_y) return b200::failed(SpMVError::INVALID_ARGUMENT);
    if (vec_size >= 0 && !spmv_validate_dimensions(A->num_cols, vec_size))
        return b200::failed(SpMVError::INVALID_DIMENSION);
    if (!A->d_row_ptrs || !A->d_col_indices || (A->nnz > 0 && !A->d_values))
        return b200::failed(SpMVError::INVALID_FORMAT);

    const int kernel = config ? static_cast<int>(config->kernel_type) : static_cast<int>(SpMVConfig::SCALAR_CSR);
    b200::ThreadCtx* ctx = b200::thread_ctx();
    if (!ctx) return b200::failed(SpMVError::KERNEL_LAUNCH);  // no usable device: fail, never compute on the host

    cudaStream_t stream = nullptr;  // legacy default stream, as the reference
    const b200::PlannedCsr* plan =
        kernel == static_cast<int>(SpMVConfig::MERGE_PATH) ? b200::auto_planned(A, stream) : nullptr;
    cudaEventRecord(ctx->start, stream);
    cudaError_t e = b200::dispatch_csr(b200::view_of(A), d_x, d_y, kernel, ctx->scratch, stream, plan);
    cudaEventRecord(ctx->stop, stream);
    cudaError_t sync = cudaEventSynchronize(ctx->stop);
    cudaError_t last = cudaGetLastError();
    if (e != cudaSuccess || sync != cudaSuccess || last != cudaSuccess)
        return b200::failed(SpMVError::KERNEL_LAUNCH);

    SpMVResult r;
    cudaEventElapsedTime(&r.elapsed_ms, ctx->start, ctx->stop);
    r.gflops = (2.0f * A->nnz) / (r.elapsed_ms * 1e6f);
    r.bandwidth_gb_s = compute_bandwidth_csr(A, r.elapsed_ms).achieved_bandwidth_gb_s;
    r.y = d_y;
    r.error_code = static_cast<int>(SpMVError::SUCCESS);
    return r;
}

// ------------------------------------------------------------------- spmv_ell --
SpMVResult spmv_ell(const ELLMatrix* A, const float* d_x, float* d_y, const SpMVConfig* /*config*/, int vec_size) {
    b200::NvtxRange nvtx_range("spmv_b200:spmv_ell");
    if (!A || !d_x || !d_y) return b200::failed(SpMVError::INVALID_ARGUMENT);
    if (vec_size >= 0 && !spmv_validate_dimensions(A->num_cols, vec_size))
        return b200::failed(SpMVError::INVALID_DIMENSION);
    if (!A->d_col_indices || !A->d_values) return b200::failed(SpMVError::INVALID_FORMAT);

    b200::ThreadCtx* ctx = b200::thread_ctx();
    if (!ctx) return b200::failed(SpMVError::KERNEL_LAUNCH);

    cudaStream_t stream = nullptr;
    cudaMemsetAsync(ctx->d_counter, 0, sizeof(unsigned long long), stream);
    cudaEventRecord(ctx->start, stream);
    cudaError_t e = b200::launch_ell(A->num_rows, A->max_nnz_per_row, A->d_col_indices, A->d_values, d_x, d_y,
                                     ctx->d_counter, stream);
    cudaEventRecord(ctx->stop, stream);
    unsigned long long live = 0;
    cudaError_t copy = cudaMemcpyAsync(&live, ctx->d_counter, sizeof(live), cudaMemcpyDeviceToHost, stream);
    cudaError_t sync = cudaStreamSynchronize(stream);
    cudaError_t last = cudaGetLastError();
    if (e != cudaSuccess || copy != cudaSuccess || sync != cudaSuccess || last != cudaSuccess)
        return b200::failed(SpMVError::KERNEL_LAUNCH);

    SpMVResult r;
    cudaEventElapsedTime(&r.elapsed_ms, ctx->start, ctx->stop);
    const int actual_nnz = static_cast<int>(live);  // entries with col >= 0 (reference :399-405)
    r.gflops = (2.0f * actual_nnz) / (r.elapsed_ms * 1e6f);
    r.bandwidth_gb_s = compute_bandwidth_ell(A, r.elapsed_ms).achieved_bandwidth_gb_s;
    r.y = d_y;
    r.error_code = static_cast<int>(SpMVError::SUCCESS);
    return r;
}

}  // namespace spmv
