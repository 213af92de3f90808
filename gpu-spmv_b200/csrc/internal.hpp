// internal.hpp -- declarations shared between the translation units of
// libspmv_b200.so.  Not installed; the public surfaces are
// include/spmv_b200/api.hpp (C++) and include/spmv_b200.h (C ABI).
#pragma once

#include "spmv_b200/api.hpp"

#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <vector>

namespace spmv {
namespace b200 {

// ---- environment ------------------------------------------------------------------
// atoi of environment variable `name`, or `fallback` when it is unset.  Callers keep the result in a
// function-local static where a variable is read once per process.
inline int env_int(const char* name, int fallback) {
    const char* v = std::getenv(name);
    return v ? std::atoi(v) : fallback;
}

// ---- selector -----------------------------------------------------------------
// A SCALAR_CSR decision is overridden to MERGE_PATH when a row is longer than
// this (one CTA of the row-owner kernel would otherwise walk it alone).
constexpr int kOutlierRowNnz = 65536;

SpMVConfig::KernelType reference_kernel_choice(const CSRStats& s);
SpMVConfig reference_policy(const CSRMatrix* A);

size_t csr_compulsory_bytes(const CSRMatrix* A);
size_t ell_compulsory_bytes(const ELLMatrix* A);

// ---- NVTX ranges (the reference has none; SURVEY 5 "tracing") ----------------------
// Header-only NVTX v3: a no-op costing one indirect call unless a tool (nsys, ncu --nvtx) is attached.
// Ranges: spmv_b200:spmv_csr / spmv_ell / spmv_csr_planned / csr_plan_create / spmv_ell_host /
// pagerank_device / pagerank_multi.run -- `ncu --nvtx --nvtx-include "spmv_b200:pagerank_device/"` profiles
// exactly the kernels of one entry point (scripts/ncu_capture.sh).
struct NvtxRange {
    explicit NvtxRange(const char* name);
    ~NvtxRange();
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

// ---- launch accounting ----------------------------------------------------------
void count_launches(int n);
unsigned long long launch_count();

// ---- device views ----------------------------------------------------------------
struct CsrView {
    int rows;
    int cols;
    int nnz;
    const int* row_ptrs;     // device [rows + 1]
    const int* col_indices;  // device [nnz]
    const float* values;     // device [nnz]
};

inline CsrView view_of(const CSRMatrix* A) {
    return CsrView{A->num_rows, A->num_cols, A->nnz, A->d_row_ptrs, A->d_col_indices, A->d_values};
}

// Grow-only device scratch (per owner; not thread-safe).
class Scratch {
public:
    Scratch() = default;
    ~Scratch();
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
    // returns nullptr on allocation failure
    void* reserve(size_t bytes);
    void release();
private:
    void* ptr_ = nullptr;
    size_t cap_ = 0;
};

// ---- merge-path geometry (shared by host planning and the kernels) ---------------
constexpr int kMergeThreads = 256;
// An ODD number of items per thread: thread t consumes products t*IPT .. t*IPT+IPT-1 from shared
// memory, and an even stride puts 4 (stride 8: 8) lanes of a warp on the same bank.  ncu on R-MAT 24
// with 8 items: half of the kernel's shared-memory wavefronts were bank-conflict replays, on the
// same L1 data pipe that serves the x gathers (profiles/r1_hub_kernel.md).
#ifndef SPMV_B200_MERGE_IPT
#define SPMV_B200_MERGE_IPT 7
#endif
constexpr int kMergeItemsPerThread = SPMV_B200_MERGE_IPT;
constexpr int kMergeTile = kMergeThreads * kMergeItemsPerThread;  // merge items per CTA

struct MergePlan {
    int num_tiles = 0;
    int2* coords = nullptr;      // [num_tiles + 1] (row, nz) at every tile diagonal
    int* carry_row = nullptr;    // [num_tiles] row left open at the tile end, or -1
    float* carry_val = nullptr;  // [num_tiles] its partial sum inside the tile
    double* partials = nullptr;  // [(num_tiles + fixup_blocks) * 3] fused-PageRank sums
    int fixup_blocks = 0;
    int ipt = kMergeItemsPerThread;  // merge items per thread of the tiles in `coords` (7, or 8 for regular matrices)
};

inline int merge_num_tiles(int rows, int nnz, int ipt = kMergeItemsPerThread) {
    const long long items = static_cast<long long>(rows) + nnz;
    const long long tile = static_cast<long long>(kMergeThreads) * ipt;
    return static_cast<int>((items + tile - 1) / tile);
}
// Items per thread of the plain MERGE_PATH tile kernel.  7 (odd: the stride-7 reads of the products are
// bank-conflict-free) wins on every skewed matrix; on short regular rows (4 <= avg < 10) 8 items = 14 % fewer tiles
// win (config 2: 0.321 against 0.380 ms).  The hub-column plan follows the same choice (bit-identity with the
// plain path); PageRank plans and the segmented stream always use 7.
int merge_items_for(int rows, int nnz);
size_t merge_plan_bytes(int rows, int nnz, bool with_partials);  // sized for 7 items (the larger tile count)
// carve a MergePlan out of a scratch block of merge_plan_bytes() bytes
MergePlan merge_plan_carve(void* block, int rows, int nnz, bool with_partials, int ipt = kMergeItemsPerThread);

// ---- fused PageRank epilogue parameters ---------------------------------------------
constexpr int kMaxPeers = 8;  // GPUs of one NVSwitch box
struct PageRankStepArgs {
    const float* r_old;     // full vector [n_global]
    float* r_new;           // full vector [n_global]
    int row_offset;         // first global row of this shard
    int n_global;
    float damping;
    float teleport;         // (1 - d) / n, or 1 - d when pvec is set; computed on the host in fp32
    const float* d_dsum;    // device scalar: dangling mass of r_old
    const uint32_t* bits;   // dangling bitmask over global node ids
    double* out;            // device [3]: sum d^2, sum |d|, next dangling mass
    // fused slice exchange: when n_peers > 1 every finished rank value is also stored into the
    // r_new buffer of every other rank (peer-mapped device pointers, NVLink), so no all-gather
    // follows the step.  peers[self_rank] is ignored (r_new is the local buffer).
    float* peers[kMaxPeers];
    int n_peers;
    int self_rank;
    // NVSwitch multicast address of r_new (NVLS): when set, ONE multimem.st per value reaches the
    // r_new buffer of every GPU of the group (this one included) instead of n_peers - 1 unicast
    // stores, so the NVLink egress of a rank is 4 bytes per owned row instead of 4 * (n_peers - 1).
    float* mc_r_new;
    // personalized PageRank: the normalised personalization vector (sums to 1) over the rows OF
    // THIS SHARD, indexed by local row (global row - row_offset).  Teleport and dangling mass are
    // spread by it instead of uniformly (dev::pr_row_value).  nullptr: global PageRank.
    const float* pvec;
};

// ---- kernel launchers (stream-ordered; return the launch status) --------------------
cudaError_t launch_ell(int rows, int width, const int* col_indices, const float* values,
                       const float* x, float* y, unsigned long long* nnz_counter,
                       cudaStream_t stream);

// Row-owner kernel: lanes_per_row == 1 is the SCALAR_CSR path (sequential
// per-row order, bit-identical to spmv_cpu_csr); 2..16 sub-warp VECTOR_CSR.
cudaError_t launch_csr_stream(const CsrView& A, const float* x, float* y, int lanes_per_row,
                              cudaStream_t stream);
// One warp per row with 128-bit loads (VECTOR_CSR for long rows).
cudaError_t launch_csr_warp_per_row(const CsrView& A, const float* x, float* y, cudaStream_t stream);
// VECTOR_CSR front end: picks lanes per row from the average row length.
cudaError_t launch_csr_vector(const CsrView& A, const float* x, float* y, cudaStream_t stream);
int vector_lanes_for(int rows, int nnz);
// longest-row cache of the row-owner launchers (csr_stream_kernels.cu), keyed by the device row_ptrs array
void seed_longest_row(const int* d_row_ptrs, int rows, int nnz, int longest);
void forget_longest_row(const int* d_row_ptrs, int rows, int nnz);

// Merge-path: partition (fills plan.coords) then tile + fix-up kernels.
cudaError_t launch_merge_partition(const CsrView& A, const MergePlan& plan, cudaStream_t stream);
cudaError_t launch_merge_spmv(const CsrView& A, const float* x, float* y, const MergePlan& plan,
                              cudaStream_t stream);
cudaError_t launch_merge_pagerank(const CsrView& A, const MergePlan& plan,
                                  const PageRankStepArgs& args, cudaStream_t stream);

// Level 3 alone (used by the tile kernel of csr_hot_kernels.cu)
cudaError_t launch_merge_fixup(const MergePlan& plan, float* y, cudaStream_t stream);
cudaError_t launch_merge_fixup_pagerank(const MergePlan& plan, const PageRankStepArgs& args, int partial_base,
                                        cudaStream_t stream);

// ---- hub-column plan (csr_hot_kernels.cu): x of the most referenced columns in shared memory ----
struct HotPlan {
    int n_hot = 0;            // columns kept in the shared-memory table (0: plan not worthwhile)
    bool all_hot = false;     // every column fits: no re-encoding, the table is x itself
    int* enc = nullptr;       // device [nnz]: col_indices with hub columns replaced by ~slot (owned)
    int* hot_cols = nullptr;  // device [n_hot]: the column of every slot (owned)
    long long hot_nnz = 0;    // non-zeros whose gather is served by the table
    int nnz = 0;
    int cols = 0;
};
int hot_capacity();                   // table slots that fit next to the tile buffers on this device
int hot_default_capacity();           // table slots used when the caller does not say (tuned, < maximum)
bool hot_worthwhile(const CsrView& A);  // large enough for the persistent grid
// Builds the plan (synchronises `stream`).  capacity <= 0: the device maximum.  Success with
// n_hot == 0 means "use the plain tile kernel".  force skips the size / benefit thresholds (tests).
// min_share: the table must serve at least nnz / min_share non-zeros for the plan to be kept.
cudaError_t hot_plan_build(const CsrView& A, HotPlan* plan, int capacity, bool force, cudaStream_t stream,
                           int min_share = 8);
// the selection step alone (shared with csr_seg_kernels.cu); see the definition
cudaError_t hot_select_columns(const CsrView& A, int capacity, int t_min, int** d_slot_of, int** d_hot_cols,
                               int* n_hot, long long* hot_nnz, cudaStream_t stream);
int device_sm_count();
void hot_plan_release(HotPlan* plan);
cudaError_t launch_hot_spmv(const CsrView& A, const HotPlan& hot, const float* x, float* y, const MergePlan& plan,
                            cudaStream_t stream);
cudaError_t launch_hot_pagerank(const CsrView& A, const HotPlan& hot, const MergePlan& plan,
                                const PageRankStepArgs& args, cudaStream_t stream);

// ---- segmented-stream plan (csr_seg_kernels.cu): row heads travel with the re-encoded stream ----
constexpr int kSegTile = 2048;  // non-zeros per tile
struct SegPlan {
    int n_hot = 0;                  // entries of the shared-memory x table (0: every gather is global)
    bool whole_x = false;           // the table is x itself (cols <= capacity)
    long long hot_nnz = 0;          // non-zeros served by the table
    int* enc = nullptr;             // device [num_tiles * kSegTile]: hub bit | head bit | slot or column
    int* hot_cols = nullptr;        // device [n_hot] column of every slot (nullptr when whole_x)
    int* rows_nz = nullptr;         // device [nonempty_rows] row of the k-th head
    int* tile_head_base = nullptr;  // device [8 * num_tiles + 1] heads before every 256-non-zero span
    uint32_t* nonempty = nullptr;   // device bit mask over rows
    float* tile_lead = nullptr;     // device [num_tiles] work arrays of a product (one product at a time)
    float* tile_tail = nullptr;
    double* partials = nullptr;     // device [3 * epilogue_blocks] PageRank sums
    int num_tiles = 0, nonempty_rows = 0, epilogue_blocks = 0;
    int rows = 0, cols = 0, nnz = 0;
    bool valid() const { return enc != nullptr; }
};
int seg_table_capacity();
int seg_default_capacity();
bool seg_worthwhile(const CsrView& A);
// Builds the plan (synchronises `stream`).  capacity <= 0: tuned default.  Success with
// !plan->valid() means "not worthwhile, use the merge-path kernels".  force skips the thresholds.
cudaError_t seg_plan_build(const CsrView& A, SegPlan* plan, int capacity, bool force, cudaStream_t stream);
void seg_plan_release(SegPlan* plan);
cudaError_t launch_seg_spmv(const CsrView& A, const SegPlan& plan, const float* x, float* y, cudaStream_t stream);
cudaError_t launch_seg_pagerank(const CsrView& A, const SegPlan& plan, const PageRankStepArgs& args, cudaStream_t stream);
// What a plan holds for the planned kernels: at most one of the two is filled.
struct PlannedCsr {
    HotPlan hot;  // scale-free matrices: hub-column merge-path kernel (csr_hot_kernels.cu)
    SegPlan seg;  // other matrices with >= 4 non-zeros per row: segmented-stream kernel (csr_seg_kernels.cu)
    bool any() const { return seg.valid() || hot.n_hot > 0; }
    void release() {
        hot_plan_release(&hot);
        seg_plan_release(&seg);
    }
};
// Chooses by measured structure (SPMV_B200_PLAN=hub|seg forces one): the hub-column plan when
// its table would serve >= 1/8 of the non-zeros, else -- if allow_seg -- the segmented-stream plan
// when rows average >= 4 non-zeros, else nothing (plain merge-path).  Synchronises `stream`.
// prefer_seg: take the segmented stream first when rows average >= 4 non-zeros (single-shard PageRank).
cudaError_t planned_build(const CsrView& A, PlannedCsr* out, int capacity, bool force, bool allow_seg,
                          cudaStream_t stream, bool prefer_seg = false);
// SPMV_B200_HOT: 0 no hub-column / segmented plans, > 0 plans without the size / benefit thresholds, -1 (unset) by structure
int hot_env_mode();
// out[3] = ordered sum of `count` triples of per-CTA partial sums
cudaError_t launch_reduce_partials(const double* partials, int count, double* out, cudaStream_t stream);

// PageRank helpers
cudaError_t launch_colsum(const CsrView& A, double* d_colsum, cudaStream_t stream);  // f64 sums: see aux_kernels.cu
cudaError_t launch_dangling_bits(const double* d_colsum, int n, int valid_cols, uint32_t* d_bits,
                                 cudaStream_t stream);
// d_tmp of launch_pr_init and launch_normalize: one double per CTA of their grids (at most 148 * 16)
constexpr int kPrScratchDoubles = 148 * 16 + 8;
cudaError_t launch_pr_init(int n, const uint32_t* d_bits, float* d_r, float* d_dsum,
                           double* d_tmp, cudaStream_t stream);
cudaError_t launch_next_dsum(const double* d_partial, float* d_dsum, cudaStream_t stream);
cudaError_t launch_normalize(const float* d_r, int n, float* d_out, double* d_tmp,
                             cudaStream_t stream);
cudaError_t launch_ell_from_csr(const CsrView& A, int width, float* ell_values, int* ell_cols,
                                cudaStream_t stream);
cudaError_t launch_max_row_len(const CsrView& A, int* d_out, cudaStream_t stream);

// ---- device-side assembly (assembly.cu) --------------------------------------------------
// (row, col, value) triplets in device memory -> device CSR sorted by (row, col), duplicates kept
// in input order; `out` receives the device arrays (csr_to_gpu ownership rules) and host arrays
// of the right size for csr_from_gpu.
int csr_from_coo_device(CSRMatrix* out, int rows, int cols, long long n_entries, const int* d_rows,
                        const int* d_cols, const float* d_vals);
// values[j] /= column sum (columns summing to 0 untouched): the column-normalised adjacency
// matrix pagerank() expects (reference include/spmv/pagerank.h:28)
int csr_normalize_columns_device(CSRMatrix* A);

// ---- device top-k of a rank vector in HBM (topk.cu); top_k is a host array of min(k, n) entries ----
int pagerank_top_k_device(const float* d_ranks, int n, int k, TopKNode* top_k);

// ---- Matrix Market coordinate files (matrix_market.cpp; host arrays only) -----------------
int csr_load_matrix_market(CSRMatrix* out, const char* filename);
int csr_save_matrix_market(const CSRMatrix* m, const char* filename);

// ---- stream-ordered dispatch used by the blocking API, benchmark and PageRank --------
// Chooses and launches the kernel(s) for `kernel_type` (any unknown value ->
// SCALAR, as src/spmv_kernels.cu:287-288).  `scratch` backs merge-path plans.
cudaError_t dispatch_csr(const CsrView& A, const float* x, float* y, int kernel_type,
                         Scratch& scratch, cudaStream_t stream, const PlannedCsr* plan = nullptr);

// ---- explicit CSR plans (dispatch.cu): merge coordinates + hub-column plan, built once ------
struct CsrPlan;
// flags: 1 = force (skip the size / benefit thresholds), 2 = the caller accepts a SNAPSHOT of the values
// (uniform matrices are then re-laid out as ELL; csr_plan_refresh_values re-reads them)
int csr_plan_create(const CSRMatrix* A, int max_hot_columns, int flags, CsrPlan** out);
int csr_plan_refresh_values(CsrPlan* plan, cudaStream_t stream);
void csr_plan_destroy(CsrPlan* plan);
void csr_plan_info(const CsrPlan* plan, int* hot_columns, long long* hot_nnz, int* mode);
int spmv_csr_planned(const CsrPlan* plan, const float* d_x, float* d_y, cudaStream_t stream);
// automatic plans of spmv_csr(MERGE_PATH) follow the device arrays uploaded by csr_to_gpu
void note_device_csr(const CSRMatrix* A);
void forget_device_csr(const void* d_col_indices);
void auto_plan_info(const CSRMatrix* A, int* hot_columns, long long* hot_nnz);
// automatic plans are opt-in (default off, or SPMV_B200_AUTO_PLAN=1): see dispatch.cu
bool auto_plan_enabled();
void set_auto_plan(bool on);

// stream-ordered twins of spmv_csr / spmv_ell (no sync, no timing); return a SpMVError
int spmv_csr_async(const CSRMatrix* A, const float* d_x, float* d_y, const SpMVConfig* config,
                   cudaStream_t stream);
int spmv_ell_async(const ELLMatrix* A, const float* d_x, float* d_y, cudaStream_t stream);

// ---- pipelined host-buffer ELL SpMV (host_pipeline.cu) -------------------------------------
struct EllHostPlan;
int ell_host_plan_create(const ELLMatrix* A, int chunks, EllHostPlan** out);
void ell_host_plan_destroy(EllHostPlan* plan);
int spmv_ell_host(EllHostPlan* plan, const float* x_host, float* y_host);
void ell_host_plan_info(const EllHostPlan* plan, int* chunks, int* ranged, int* max_lookahead);
void ell_host_plan_bytes(const EllHostPlan* plan, unsigned long long* h2d, unsigned long long* d2h);
void ell_host_plan_gated(const EllHostPlan* plan, int* gated, int* down_chunks);
int probe_h2d_order(const float* x_host, size_t n, int samples, long long* out_ns, int mode, unsigned sleep_ns);

// ---- PageRank plan over one row shard (pagerank.cu) -------------------------------------
struct PrPlan;
int pr_plan_create(const CSRMatrix* shard, int row_offset, int n_global, cudaStream_t stream, PrPlan** out);
void pr_plan_destroy(PrPlan* plan);
int pr_plan_set_hot(PrPlan* plan, int max_hot_columns, bool force, cudaStream_t stream);
// d_pvec: this shard's rows of the normalised personalization vector (PageRankStepArgs::pvec), or nullptr
int pr_step(PrPlan* plan, const float* d_r_old, float* d_r_new, float damping, const float* d_dsum,
            const uint32_t* d_bits, double* d_partial, cudaStream_t stream,
            float* const* peer_r_new = nullptr, int n_peers = 0, int self_rank = 0, float* mc_r_new = nullptr,
            const float* d_pvec = nullptr);
const CsrView& pr_plan_view(const PrPlan* plan);
int pr_plan_hub_columns(const PrPlan* plan);  // entries of the shared-memory x table in use (0: none)
double* pr_plan_tmp(PrPlan* plan);
// Dangling bitmask of a whole graph (A.rows == A.cols): zeroes d_colsum [A.cols], sums the columns into it in f64 and
// sets bit c where column c sums to 0 (reference src/pagerank.cu:20-48).
cudaError_t pr_dangling_bits(const CsrView& A, double* d_colsum, uint32_t* d_bits, cudaStream_t stream);

// CUDA graphs of the two ping-pong iterations of a PageRank loop (p = 0: vector a -> b, p = 1: b -> a), captured
// once and replayed: one graph launch per iteration instead of one API call per kernel and copy, where small graphs
// are launch-bound.  SPMV_B200_PR_GRAPH=0 disables them.
struct PrIterationGraphs {
    cudaGraphExec_t exec[2] = {nullptr, nullptr};
    unsigned long long launches_per_iteration = 0;  // launches one replay stands for (set by capture)
    PrIterationGraphs() = default;
    PrIterationGraphs(const PrIterationGraphs&) = delete;
    PrIterationGraphs& operator=(const PrIterationGraphs&) = delete;
    ~PrIterationGraphs() { reset(); }
    // capturing pays off for a loop of this many iterations (and SPMV_B200_PR_GRAPH allows it)
    static bool wanted(int iterations);
    bool ready() const { return exec[0] && exec[1]; }
    // enqueue(p) enqueues iteration p on `stream` and returns 0.  On any failure no graph is kept, false is
    // returned, and launch_count() is what it was before the call.
    bool capture(cudaStream_t stream, const std::function<int(int)>& enqueue);
    // replays iteration p and counts its launches
    bool launch(int p, cudaStream_t stream);
    void reset();
};
// d_pvec: the normalised personalization vector [n] on the device (pr_personalization_upload), or nullptr
int pagerank_device(const CSRMatrix* adj, const PageRankConfig* config, float* d_ranks, int* iterations,
                    float* final_residual, bool* converged, double* l1_residual, bool normalize = true, float* l2_history = nullptr, int history_capacity = 0,
                    const float* d_pvec = nullptr);
// pagerank()'s body: host ranks in *result (new[]; nullptr on a failed validation).  personalization: host [n]
// or nullptr (global PageRank, exactly pagerank()).  Returns INVALID_ARGUMENT for a rejected personalization.
int pagerank_to_host(const CSRMatrix* adj, const PageRankConfig* config, const float* personalization,
                     PageRankResult* result);
// Personalization vector v (host, n entries): rejected (INVALID_ARGUMENT) when an entry is NaN, +-Inf or
// negative, or when the f64 sum of the entries, in index order, is 0.  vhat[i] = (float)((double)v[i] / sum).
// Host code only: every rank of a sharded run computes the same vhat from the same v.
int pr_personalization_normalise(const float* v, int n, std::vector<float>* vhat);
// Validates and normalises v as above, then copies rows [row_lo, row_lo + rows) of vhat into a new device
// buffer of max(rows, 1) floats (*d_out; cudaFree it), complete on return (`stream` is synchronised).
// v == nullptr: *d_out = nullptr, success.
int pr_personalization_upload(const float* v, int n, int row_lo, int rows, float** d_out, cudaStream_t stream);

}  // namespace b200
}  // namespace spmv
