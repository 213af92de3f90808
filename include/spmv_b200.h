/*
 * spmv_b200.h -- C ABI of the B200-native SpMV library (libspmv_b200.so).
 *
 * This is the FFI boundary: extern "C", plain pointers and sizes, POD structs,
 * int status codes, no C++ or torch types.  Every entry point is the C twin of
 * one function of the LessUp/gpu-spmv C++ API and cites the reference
 * declaration it replaces (paths relative to the reference repository).  The
 * structs are layout-identical to the reference's (`spmv::CSRMatrix` ==
 * `spmv_b200_csr`, ...), so a pointer obtained from the C++ surface
 * (include/spmv_b200/api.hpp) can be passed here and vice versa.
 *
 * Conventions
 *   - status: 0 or a negative spmv_b200_status (include/spmv/common.h:13-23).
 *   - by-value C++ results (SpMVResult, PageRankResult, BenchmarkResult ...)
 *     become out-parameters.
 *   - nothing throws across this boundary.
 *   - d_* / "device" pointers must be valid on the CURRENT CUDA device.
 *   - there is no CPU fallback: device entry points fail with a CUDA status
 *     when no sm_100 device is usable.
 *
 * Section E (extensions) is additive: stream-ordered calls, device-resident
 * PageRank, row-sharded building blocks for one-process-per-GPU runs.
 */
#ifndef SPMV_B200_H
#define SPMV_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPMV_B200_API __attribute__((visibility("default")))

/* ---- status codes: include/spmv/common.h:13-23 ---- */
typedef enum spmv_b200_status {
    SPMV_B200_SUCCESS = 0,
    SPMV_B200_INVALID_DIMENSION = -1,
    SPMV_B200_CUDA_MALLOC = -2,
    SPMV_B200_CUDA_MEMCPY = -3,
    SPMV_B200_KERNEL_LAUNCH = -4,
    SPMV_B200_INVALID_FORMAT = -5,
    SPMV_B200_FILE_IO = -6,
    SPMV_B200_OUT_OF_MEMORY = -7,
    SPMV_B200_INVALID_ARGUMENT = -8
} spmv_b200_status;

/* include/spmv/common.h:26-39 */
SPMV_B200_API const char* spmv_b200_error_string(int status);

/* ---- POD structs ---- */

/* include/spmv/csr_matrix.h:11-28 (72 bytes) */
typedef struct spmv_b200_csr {
    int num_rows, num_cols, nnz;
    float* values;
    int* col_indices;
    int* row_ptrs;
    float* d_values;
    int* d_col_indices;
    int* d_row_ptrs;
    bool owns_host_memory;
    bool owns_device_memory;
} spmv_b200_csr;

/* include/spmv/csr_matrix.h:64-69 */
typedef struct spmv_b200_csr_stats {
    float avg_nnz_per_row;
    int max_nnz_per_row;
    int min_nnz_per_row;
    float skewness;
} spmv_b200_csr_stats;

/* include/spmv/ell_matrix.h:13-29 (56 bytes) */
typedef struct spmv_b200_ell {
    int num_rows, num_cols, max_nnz_per_row;
    float* values;
    int* col_indices;
    float* d_values;
    int* d_col_indices;
    bool owns_host_memory;
    bool owns_device_memory;
} spmv_b200_ell;

/* include/spmv/spmv.h:13-18 */
enum {
    SPMV_B200_SCALAR_CSR = 0,
    SPMV_B200_VECTOR_CSR = 1,
    SPMV_B200_MERGE_PATH = 2,
    SPMV_B200_ELL_KERNEL = 3
};

/* include/spmv/spmv.h:11-24 (12 bytes) */
typedef struct spmv_b200_config {
    int kernel_type;
    int block_size;
    bool use_texture;
} spmv_b200_config;

/* include/spmv/spmv.h:27-36 (24 bytes) */
typedef struct spmv_b200_result {
    float* y;
    float elapsed_ms;
    float gflops;
    float bandwidth_gb_s;
    int error_code;
} spmv_b200_result;

/* include/spmv/bandwidth.h:10-18 */
typedef struct spmv_b200_bandwidth {
    float theoretical_bandwidth_gb_s;
    float achieved_bandwidth_gb_s;
    float efficiency;
} spmv_b200_bandwidth;

/* include/spmv/pagerank.h:9-15 */
typedef struct spmv_b200_pagerank_config {
    float damping_factor;
    float tolerance;
    int max_iterations;
} spmv_b200_pagerank_config;

/* include/spmv/pagerank.h:18-25 (24 bytes) */
typedef struct spmv_b200_pagerank_result {
    float* ranks;
    int iterations;
    float final_residual;
    bool converged;
} spmv_b200_pagerank_result;

/* include/spmv/pagerank.h:35-38 */
typedef struct spmv_b200_topk_node {
    int node_id;
    float rank;
} spmv_b200_topk_node;

/* include/spmv/benchmark.h:34-40 */
typedef struct spmv_b200_bench_config {
    int num_warmup_runs;
    int num_runs;
    bool compare_cpu;
} spmv_b200_bench_config;

/* C-safe image of include/spmv/benchmark.h:13-31 (std::string -> char[64]) */
typedef struct spmv_b200_bench_result {
    char name[64];
    float execution_time_ms;
    float gflops;
    float bandwidth_gb_s;
    float avg_time_ms;
    float min_time_ms;
    float max_time_ms;
    float stddev_time_ms;
    int num_runs;
} spmv_b200_bench_result;

/* ======================================================================= */
/* A. CSR storage -- include/spmv/csr_matrix.h:31-71                        */
/* ======================================================================= */
SPMV_B200_API spmv_b200_csr* spmv_b200_csr_create(int rows, int cols, int nnz);          /* :31 */
SPMV_B200_API void spmv_b200_csr_destroy(spmv_b200_csr* mat);                             /* :34 */
SPMV_B200_API int spmv_b200_csr_from_dense(spmv_b200_csr* csr, const float* dense,
                                           int rows, int cols);                          /* :39 */
SPMV_B200_API int spmv_b200_csr_to_dense(const spmv_b200_csr* csr, float* dense);         /* :43 */
SPMV_B200_API float spmv_b200_csr_get_element(const spmv_b200_csr* mat, int row, int col); /* :46 */
SPMV_B200_API int spmv_b200_csr_to_gpu(spmv_b200_csr* mat);                               /* :49 */
SPMV_B200_API int spmv_b200_csr_from_gpu(spmv_b200_csr* mat);                             /* :52 */
SPMV_B200_API void spmv_b200_csr_free_gpu(spmv_b200_csr* mat);                            /* :55 */
SPMV_B200_API int spmv_b200_csr_serialize(const spmv_b200_csr* mat, const char* filename);/* :58 */
SPMV_B200_API int spmv_b200_csr_deserialize(spmv_b200_csr* mat, const char* filename);    /* :61 */
SPMV_B200_API int spmv_b200_csr_compute_stats(const spmv_b200_csr* mat,
                                              spmv_b200_csr_stats* out);                 /* :71 */

/* ======================================================================= */
/* B. ELL storage -- include/spmv/ell_matrix.h:31-66                        */
/* ======================================================================= */
SPMV_B200_API spmv_b200_ell* spmv_b200_ell_create(int rows, int cols, int max_nnz_per_row); /* :32 */
SPMV_B200_API void spmv_b200_ell_destroy(spmv_b200_ell* mat);                              /* :35 */
SPMV_B200_API int spmv_b200_ell_from_dense(spmv_b200_ell* ell, const float* dense,
                                           int rows, int cols);                           /* :38 */
SPMV_B200_API int spmv_b200_ell_from_csr(spmv_b200_ell* ell, const spmv_b200_csr* csr);    /* :41 */
SPMV_B200_API int spmv_b200_ell_to_dense(const spmv_b200_ell* ell, float* dense);          /* :44 */
SPMV_B200_API float spmv_b200_ell_get_element(const spmv_b200_ell* mat, int row, int col); /* :47 */
SPMV_B200_API int spmv_b200_ell_to_gpu(spmv_b200_ell* mat);                                /* :50 */
SPMV_B200_API int spmv_b200_ell_from_gpu(spmv_b200_ell* mat);                              /* :53 */
SPMV_B200_API void spmv_b200_ell_free_gpu(spmv_b200_ell* mat);                             /* :56 */
SPMV_B200_API int spmv_b200_ell_serialize(const spmv_b200_ell* mat, const char* filename); /* :59 */
SPMV_B200_API int spmv_b200_ell_deserialize(spmv_b200_ell* mat, const char* filename);     /* :62 */
SPMV_B200_API int spmv_b200_ell_index(int row, int k, int num_rows);                       /* :64-66 */

/* ======================================================================= */
/* C. SpMV + selector -- include/spmv/spmv.h:39-54                          */
/* ======================================================================= */
/* host reference functions of the API (never used by the device path) */
SPMV_B200_API void spmv_b200_spmv_cpu_csr(const spmv_b200_csr* A, const float* x, float* y); /* :39 */
SPMV_B200_API void spmv_b200_spmv_cpu_ell(const spmv_b200_ell* A, const float* x, float* y); /* :40 */

/* device SpMV, blocking; config may be NULL (defaults {SCALAR_CSR,256,false});
 * vec_size < 0 skips the dimension check.  Returns out->error_code. */
SPMV_B200_API int spmv_b200_spmv_csr(const spmv_b200_csr* A, const float* d_x, float* d_y,
                                     const spmv_b200_config* config, int vec_size,
                                     spmv_b200_result* out);                              /* :43-44 */
SPMV_B200_API int spmv_b200_spmv_ell(const spmv_b200_ell* A, const float* d_x, float* d_y,
                                     const spmv_b200_config* config, int vec_size,
                                     spmv_b200_result* out);                              /* :45-46 */
SPMV_B200_API int spmv_b200_auto_config(const spmv_b200_csr* A, spmv_b200_config* out);    /* :49 */
SPMV_B200_API bool spmv_b200_validate_dimensions(int num_cols, int vec_size);              /* :52-54 */

/* ======================================================================= */
/* D. Bandwidth model, PageRank, benchmark harness                          */
/* ======================================================================= */
SPMV_B200_API int spmv_b200_bandwidth_csr(const spmv_b200_csr* A, float elapsed_ms,
                                          spmv_b200_bandwidth* out);   /* bandwidth.h:21 */
SPMV_B200_API int spmv_b200_bandwidth_ell(const spmv_b200_ell* A, float elapsed_ms,
                                          spmv_b200_bandwidth* out);   /* bandwidth.h:24 */
SPMV_B200_API float spmv_b200_peak_bandwidth(void);                    /* bandwidth.h:27 */

/* config may be NULL ({0.85, 1e-6, 100}).  out->ranks is a host array owned by
 * the library; release with spmv_b200_pagerank_free. */
SPMV_B200_API int spmv_b200_pagerank(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                     spmv_b200_pagerank_result* out);  /* pagerank.h:29-32 */
SPMV_B200_API void spmv_b200_pagerank_free(spmv_b200_pagerank_result* result); /* pagerank.h:35 */
SPMV_B200_API int spmv_b200_pagerank_top_k(const spmv_b200_pagerank_result* result, int num_nodes,
                                           int k, spmv_b200_topk_node* top_k); /* pagerank.h:43 */

/* x is a HOST vector; A must already be on the device (benchmark.h:43-56) */
SPMV_B200_API int spmv_b200_benchmark_csr(const spmv_b200_csr* A, const float* x,
                                          const spmv_b200_config* config,
                                          const spmv_b200_bench_config* bench_config,
                                          spmv_b200_bench_result* out);          /* benchmark.h:43 */
SPMV_B200_API int spmv_b200_benchmark_ell(const spmv_b200_ell* A, const float* x,
                                          const spmv_b200_bench_config* bench_config,
                                          spmv_b200_bench_result* out);          /* benchmark.h:51 */
SPMV_B200_API int spmv_b200_compare_gpu_cpu_csr(const spmv_b200_csr* A, const float* x,
                                                const spmv_b200_config* config,
                                                const spmv_b200_bench_config* bench_config,
                                                spmv_b200_bench_result* gpu_out,
                                                spmv_b200_bench_result* cpu_out,
                                                float* speedup);                 /* benchmark.h:66 */
/* returns the JSON length (excluding NUL) or -1 when cap is too small */
SPMV_B200_API int spmv_b200_benchmark_to_json(const spmv_b200_bench_result* result,
                                              char* buf, int cap);               /* benchmark.h:74 */
SPMV_B200_API int spmv_b200_benchmark_from_json(const char* json,
                                                spmv_b200_bench_result* out);    /* benchmark.h:78 */

/* Roofline-aware report of the same measurement (additive; the byte format of benchmark_to_json is
 * pinned by the reference's round-trip test, tests/test_benchmark.cu:151-170, so the extra figures
 * get their own writer).  Runs benchmark_csr (benchmark.h:43) and, when bench_config->compare_cpu is
 * set, times spmv_cpu_csr on the host like compare_gpu_cpu_csr (src/benchmark.cu:151-167).  The JSON
 * object holds the reference's nine keys (same names, same formatting) followed by
 *   "kernel"                selector decision or the caller's choice (SCALAR_CSR, ...)
 *   "algorithmic_bytes"     8*nnz + 4*(rows+1) + 4*cols + 4*rows  (src/bandwidth.cpp:34-42)
 *   "effective_gb_s"        algorithmic_bytes / avg_time_ms
 *   "peak_gb_s"             peak_gb_s argument, or (<= 0) the device's theoretical HBM bandwidth
 *   "roofline_fraction"     effective_gb_s / peak_gb_s
 *   "cpu_avg_time_ms", "cpu_threads" (1: the reference's CPU path is single-threaded), "speedup"
 * Returns the JSON length (excluding NUL), -1 when cap is too small, or a negative status. */
SPMV_B200_API int spmv_b200_benchmark_csr_report(const spmv_b200_csr* A, const float* x,
                                                 const spmv_b200_config* config,
                                                 const spmv_b200_bench_config* bench_config,
                                                 float peak_gb_s, char* buf, int cap);

/* ======================================================================= */
/* E. Extensions (additive; nothing in the reference corresponds)           */
/* ======================================================================= */

SPMV_B200_API const char* spmv_b200_version(void);
/* cudaLimitMaxL2FetchGranularity of the current device (32, 64 or 128 bytes; a hint the driver may
 * round): a product whose x does not fit L2 (config 3: 200 MB of x behind random columns) pays DRAM for
 * every gather, and at the default granularity each 4-byte gather fetches 64 bytes.  get returns the
 * current value or a negative status. */
SPMV_B200_API int spmv_b200_set_l2_fetch_granularity(int bytes);
SPMV_B200_API int spmv_b200_get_l2_fetch_granularity(void);
/* L2 persistence for the x of products whose x does not fit L2 (design probe, profiles/r2_l2_persist.jsonl): reserve
 * set_aside_bytes of L2 for persisting lines (cudaLimitPersistingL2CacheSize) and give `stream` an access-policy window
 * over [base, base + bytes): a hit_ratio share of its lines persists, the rest streams.  base == NULL removes the window
 * and resets the persisting lines.  limits: the device's maximum set-aside, maximum window and L2 size. */
SPMV_B200_API int spmv_b200_l2_persistence_limits(unsigned long long* max_set_aside_bytes, unsigned long long* max_window_bytes,
                                                  unsigned long long* l2_bytes);
SPMV_B200_API int spmv_b200_set_l2_persistence(void* stream, const void* base, unsigned long long bytes, float hit_ratio,
                                               unsigned long long set_aside_bytes);
/* number of kernels this library has launched in this process so far */
SPMV_B200_API unsigned long long spmv_b200_launch_count(void);
/* the reference's selector decision without the B200 outlier override
 * (src/spmv_cpu.cpp:34-50 verbatim); spmv_b200_auto_config == this unless the
 * matrix has avg < 4 AND a row longer than 65536 nnz (then MERGE_PATH). */
SPMV_B200_API int spmv_b200_reference_policy(const spmv_b200_csr* A, spmv_b200_config* out);

/* stream-ordered SpMV: no sync, no timing.  stream is a cudaStream_t. */
SPMV_B200_API int spmv_b200_spmv_csr_async(const spmv_b200_csr* A, const float* d_x, float* d_y,
                                           const spmv_b200_config* config, void* stream);
SPMV_B200_API int spmv_b200_spmv_ell_async(const spmv_b200_ell* A, const float* d_x, float* d_y,
                                           void* stream);

/* ---- host-buffer SpMV, overlapped -----------------------------------------
 * y_host = A x_host for an ELL matrix resident on the device while x and y live in HOST memory:
 * what a caller of the reference writes as cudaMemcpy(x) + spmv_ell + cudaMemcpy(y)
 * (reference README.md:98-118, src/benchmark.cu:36-38,95-102), with the upload of x, the product
 * and the way down of y overlapped.  Two forms (spmv_b200_ell_host_plan_gated below tells which):
 * the GATED form -- one upload, one persistent kernel that consumes x while it arrives; the default
 * for matrices the TMA ring covers -- and the CHUNKED form -- upload, product and download pipelined
 * over `chunks` row chunks on three streams; the plan measures, once, which x entries every row chunk
 * reads (its column range), so a banded matrix overlaps the PCIe up- and down-link, any other matrix
 * degenerates to upload, then compute overlapped with the download.  y is bit-identical to spmv_ell
 * in both.  The matrix's device arrays are borrowed and must outlive the plan.  chunks <= 0: 12.
 * x_host / y_host should be page-locked (with a page-locked y_host the kernels store y straight into it). */
typedef struct spmv_b200_ell_host_plan spmv_b200_ell_host_plan;
SPMV_B200_API int spmv_b200_ell_host_plan_create(const spmv_b200_ell* A, int chunks,
                                                 spmv_b200_ell_host_plan** out);
SPMV_B200_API void spmv_b200_ell_host_plan_destroy(spmv_b200_ell_host_plan* plan);
/* blocking: returns when y_host is complete */
SPMV_B200_API int spmv_b200_spmv_ell_host(spmv_b200_ell_host_plan* plan, const float* x_host,
                                          float* y_host);
/* chunks in use; whether the row-range kernel applies; the largest number of x chunks beyond its
 * own index any row chunk has to wait for (0-1 for a banded matrix, chunks - 1 in the worst case) */
SPMV_B200_API int spmv_b200_ell_host_plan_info(const spmv_b200_ell_host_plan* plan, int* chunks,
                                               int* ranged, int* max_lookahead);
/* bytes one call moves over PCIe: only the x chunks some row of the matrix reads are uploaded (a row
 * shard of a larger system reads its own band of x), plus all of y */
SPMV_B200_API int spmv_b200_ell_host_plan_bytes(const spmv_b200_ell_host_plan* plan,
                                                unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);

/* Whether the next call takes the GATED form, and how many row chunks a download by copies would use.  Gated =
 * one upload copy over a device x pre-filled with a sentinel bit pattern and ONE persistent kernel that consumes x
 * while it arrives (a 256-row window starts when the last x entry it reads is no longer the sentinel; every gather
 * is checked, so the result never depends on the order in which the copy lands).  With a page-locked (device-
 * mapped) y_host the kernel stores y straight into it and nothing is copied down; any other y_host is downloaded
 * in *down_chunks D2H copies, each queued by the calling thread when the kernel reports the chunk complete.
 * SPMV_B200_HOST_GATED=0 selects the chunked form (one upload / launch per row chunk); a call whose x does not
 * arrive within SPMV_B200_HOST_GATED_TIMEOUT_MS repeats itself in the chunked form and the plan stays there.
 * An x that really contains the sentinel pattern (0x7FA3C0DE, a signalling NaN) is handled correctly, only later
 * (such entries are accepted when the upload is complete). */
SPMV_B200_API int spmv_b200_ell_host_plan_gated(const spmv_b200_ell_host_plan* plan, int* gated, int* down_chunks);

/* Diagnostic behind the gated form's design: the ORDER in which one host-to-device copy of n floats lands in
 * device memory.  out_ns[i] = arrival time (ns, relative to the earliest) of entry i * (n / samples), observed by
 * a kernel that polls a sentinel-filled destination while the copy engine writes it (mode 0 / 1 / 2: system-scope /
 * gpu-scope / volatile loads, sleep_ns between polls; mode < 0: no polling); out_ns[samples] = duration of the copy by
 * CUDA events, so out_ns holds samples + 1 values.  samples <= 4096. */
SPMV_B200_API int spmv_b200_probe_h2d_order(const float* x_host, unsigned long long n, int samples, long long* out_ns,
                                            int mode, unsigned sleep_ns);

/* device-side ELL assembly from the DEVICE arrays of csr (ell_from_csr
 * semantics, src/ell_matrix.cpp:111-159); fills ell's device arrays only
 * (allocates them, sets owns_device_memory) and dims. */
SPMV_B200_API int spmv_b200_ell_from_csr_device(spmv_b200_ell* ell, const spmv_b200_csr* csr);

/* canonical merge-path coordinate of one diagonal (host; what the partition
 * kernel computes per tile) and the nnz-balanced row split used for sharding */
SPMV_B200_API int spmv_b200_merge_path_search(int diagonal, const int* row_ptrs, int num_rows,
                                              int nnz, int* out_row, int* out_nz);
SPMV_B200_API int spmv_b200_partition_rows(const int* row_ptrs, int num_rows, int parts,
                                           int* bounds /* [parts+1] */);
/* the same split with the work of a row counted as nnz + row_weight (row_weight = 1 balances the
 * merge-path items rows + nnz, which is what the merge-path / PageRank kernels consume) */
SPMV_B200_API int spmv_b200_partition_rows_weighted(const int* row_ptrs, int num_rows, int parts,
                                                    int row_weight, int* bounds /* [parts+1] */);

/* ---- device top-k (SURVEY 8f rank 4) ---------------------------------------- */

/* Top-k of a rank vector that is already in device memory (e.g. spmv_b200_pagerank_device's
 * d_ranks): radix select + ordered tie fill on the device, only min(k, n) pairs are downloaded.
 * Same values as pagerank_top_k (src/pagerank.cu:162-185, which sorts a host copy of all n
 * pairs); equal ranks are ordered by ascending node id (the reference leaves ties unordered). */
SPMV_B200_API int spmv_b200_pagerank_top_k_device(const float* d_ranks, int num_nodes, int k,
                                                  spmv_b200_topk_node* top_k);

/* ---- Matrix Market input (SURVEY 8f rank 4) ------------------------------- */

/* `%%MatrixMarket matrix coordinate {real|integer|pattern} {general|symmetric|skew-symmetric}`
 * -> host arrays of `out` (re-allocated and owned, sorted by (row, column), symmetric files
 * expanded, pattern entries = 1, duplicates kept in file order; device arrays untouched, as
 * csr_from_dense, src/csr_matrix.cpp:50-95).  The reference lists real-matrix input as a
 * requirement but has no loader.  Unreadable file -> FILE_IO; anything else unsupported or
 * malformed -> INVALID_FORMAT with `out` unchanged. */
SPMV_B200_API int spmv_b200_csr_load_matrix_market(spmv_b200_csr* out, const char* filename);
/* coordinate real general, CSR order, values with 9 significant digits (exact for fp32) */
SPMV_B200_API int spmv_b200_csr_save_matrix_market(const spmv_b200_csr* m, const char* filename);

/* ---- device-side assembly (SURVEY 8f rank 1) ------------------------------ */

/* (row, col, value) triplets in DEVICE memory -> CSR sorted by (row, col) in the device arrays of
 * `out` (allocated here, owns_device_memory = true; duplicates are kept, in input order).  The
 * reference can only assemble from a dense host array (csr_from_dense, src/csr_matrix.cpp:50-95).
 * Host arrays of `out` are re-allocated to the new size (uninitialised) so that csr_from_gpu can
 * fill them.  An index outside [0, rows) x [0, cols) -> INVALID_ARGUMENT, nothing is changed. */
SPMV_B200_API int spmv_b200_csr_from_coo_device(spmv_b200_csr* out, int rows, int cols,
                                                long long n_entries, const int* d_row_indices,
                                                const int* d_col_indices, const float* d_values);
/* d_values[j] /= sum of column d_col_indices[j] (columns summing to 0 are left alone): the
 * column-normalised adjacency matrix pagerank() expects (include/spmv/pagerank.h:28). */
SPMV_B200_API int spmv_b200_csr_normalize_columns_device(spmv_b200_csr* A);

/* ---- CSR plans: merge coordinates + hub-column table, built once --------- */

/*
 * Opaque plan over the DEVICE arrays of a CSR matrix for repeated MERGE_PATH products with the
 * same sparsity pattern (the "persistent workspace" the reference lacks: its spmv_csr recomputes
 * everything per call, src/spmv_kernels.cu:258-297).  It holds (1) the merge-path tile
 * coordinates and (2) a PRIVATE re-encoding of col_indices for one of the two planned kernels,
 * chosen by the measured structure: scale-free matrices (a table of the max_hot_columns most
 * referenced columns would serve >= 1/8 of the non-zeros) get the hub-column merge-path kernel of
 * csr_hot_kernels.cu, which keeps those x entries in shared memory; other matrices with >= 4
 * non-zeros per row get the segmented-stream kernel of csr_seg_kernels.cu, whose re-encoding also
 * carries the row starts.  The caller's arrays are not modified;
 * d_values is read live at every product, d_row_ptrs / d_col_indices must not change while the
 * plan is alive.  max_hot_columns <= 0: the tuned default (24576 on B200; the table competes with
 * the L1 for the same 256 KB).  flags: SPMV_B200_PLAN_* below.  A plan owns the work arrays of a product, so it serves ONE product at
 * a time: use one plan per stream (or order the products).
 */
typedef struct spmv_b200_csr_plan spmv_b200_csr_plan;
#define SPMV_B200_PLAN_FORCE 1            /* skip the size / benefit thresholds (tests) */
#define SPMV_B200_PLAN_SNAPSHOT_VALUES 2  /* see below */
SPMV_B200_API int spmv_b200_csr_plan_create(const spmv_b200_csr* A, int max_hot_columns, int flags,
                                            spmv_b200_csr_plan** out);
/* With SPMV_B200_PLAN_SNAPSHOT_VALUES the caller allows the plan to keep its own copy of the VALUES:
 * a uniform matrix (longest row <= 8 and rows * longest <= 1.125 * nnz) is then re-laid out as
 * column-major ELL on the device (ell_from_csr semantics, src/ell_matrix.cpp:111-159) and multiplied
 * by the ELL kernel -- the routing the reference's ELL_KERNEL enumerator promises but
 * spmv_auto_config never performs (spmv.h:16, src/spmv_cpu.cpp:41-47); mode 5, bit-identical to
 * SCALAR_CSR / spmv_cpu_csr.  After changing d_values call this to re-read them (stream-ordered;
 * a no-op for the other modes, which read d_values live). */
SPMV_B200_API int spmv_b200_csr_plan_refresh_values(spmv_b200_csr_plan* plan, void* stream);
SPMV_B200_API void spmv_b200_csr_plan_destroy(spmv_b200_csr_plan* plan);
/* hot_columns: table entries in use; hot_nnz: non-zeros served by the table;
 * mode: 0 plain merge-path tile kernel with precomputed coordinates,
 *       1 hub-column merge-path kernel, 2 the same with the whole x in the table,
 *       3 segmented-stream kernel (csr_seg_kernels.cu), 4 the same with the whole x in the table,
 *       5 ELL layout + ELL kernel (only with SPMV_B200_PLAN_SNAPSHOT_VALUES) */
SPMV_B200_API int spmv_b200_csr_plan_info(const spmv_b200_csr_plan* plan, int* hot_columns,
                                          long long* hot_nnz, int* mode);
/* y = A x through the plan; stream-ordered (stream is a cudaStream_t), no sync, no timing.
 * Deterministic; modes 0-2 are bit-identical to spmv_csr(MERGE_PATH), modes 3-4 sum in a
 * different (fixed) order and agree within the fp32 SpMV tolerance. */
SPMV_B200_API int spmv_b200_spmv_csr_planned(const spmv_b200_csr_plan* plan, const float* d_x,
                                             float* d_y, void* stream);
/* OPT-IN automatic plans (off by default; also SPMV_B200_AUTO_PLAN=1): when enabled,
 * spmv_csr(MERGE_PATH) attaches such a plan by itself to device arrays uploaded by csr_to_gpu, from
 * the second call on.  Off by default because the reference's d_col_indices / d_row_ptrs fields are
 * public and may legally be rewritten in place (reference include/spmv/csr_matrix.h:11-28): a plan
 * keeps a private re-encoding of both, so results would silently follow the OLD pattern.  A caller
 * that enables it must call spmv_b200_csr_forget_plan after such an edit (csr_to_gpu / csr_free_gpu /
 * csr_destroy drop the plan themselves).  Costs 4 B of device memory per non-zero. */
SPMV_B200_API void spmv_b200_set_auto_plan(int enabled);
SPMV_B200_API int spmv_b200_auto_plan_enabled(void);
SPMV_B200_API void spmv_b200_csr_forget_plan(const spmv_b200_csr* A);
/* the automatic plan currently attached to A's device arrays (hot_columns == 0: none) */
SPMV_B200_API int spmv_b200_csr_auto_plan_info(const spmv_b200_csr* A, int* hot_columns,
                                               long long* hot_nnz);

/* ---- device-resident PageRank building blocks --------------------------- */

/* Opaque plan over ONE row shard of an n_global x n_global column-normalised
 * matrix: rows [row_offset, row_offset + shard->num_rows), global column ids,
 * device arrays only.  Single GPU == one shard with row_offset 0. */
typedef struct spmv_b200_pr_plan spmv_b200_pr_plan;

SPMV_B200_API int spmv_b200_pr_plan_create(const spmv_b200_csr* shard, int row_offset,
                                           int n_global, void* stream, spmv_b200_pr_plan** out);
SPMV_B200_API void spmv_b200_pr_plan_destroy(spmv_b200_pr_plan* plan);
/* The plan carries the hub-column table of its shard when that pays (see spmv_b200_csr_plan).
 * This call rebuilds it: max_hot_columns 0 = none (plain tile kernel), < 0 = device maximum.
 * Returns the number of hub columns now in use (>= 0) or a negative status. */
SPMV_B200_API int spmv_b200_pr_plan_set_hot(spmv_b200_pr_plan* plan, int max_hot_columns, int force,
                                            void* stream);

/* d_colsum[c] += sum of this shard's values in column c; f64 accumulators: a sum that is never
 * rounded does not depend on the order of the atomics, so the dangling set is deterministic */
SPMV_B200_API int spmv_b200_pr_colsum(const spmv_b200_pr_plan* plan, double* d_colsum, void* stream);
/* d_bits[c/32] bit c%32 = ((float)d_colsum[c] == 0.0f)  (dangling columns) */
SPMV_B200_API int spmv_b200_pr_dangling_bits(const double* d_colsum, int n, uint32_t* d_bits,
                                             void* stream);
/* d_r[i] = 1.0f / n for the whole vector; d_dsum[0] = mass on dangling nodes */
SPMV_B200_API int spmv_b200_pr_init(int n, const uint32_t* d_bits, float* d_r, float* d_dsum,
                                    void* stream);
/*
 * One fused iteration on this shard (SpMV + damping/teleport + dangling
 * contribution + residuals + next dangling mass in one pass):
 *   r_new[row_offset + i] = (d * (A r_old)[i] + d * dsum / n) + (1 - d) / n
 *   d_partial[0] += sum (r_new - r_old)^2   (f64)
 *   d_partial[1] += sum |r_new - r_old|     (f64)
 *   d_partial[2] += sum over dangling rows of r_new  (f64)
 * d_r_old / d_r_new are FULL n_global-length vectors; d_dsum points to the
 * dangling mass of r_old (fp32, device).  d_partial is overwritten with this
 * shard's three sums (deterministic order).
 */
SPMV_B200_API int spmv_b200_pr_step(spmv_b200_pr_plan* plan, const float* d_r_old, float* d_r_new,
                                    float damping, const float* d_dsum, const uint32_t* d_bits,
                                    double* d_partial /* [3] */, void* stream);
/*
 * The same step with the slice exchange FUSED into it (one process per GPU on an
 * NVLink/NVSwitch box): peer_r_new is a host array of n_peers device pointers, entry p being
 * rank p's r_new buffer mapped into this process (spmv_b200_ipc_open); every finished rank value
 * is stored into all of them from inside the kernel, tile by tile, so no all-gather follows.
 * The caller must order the next iteration after all ranks' steps (the all-reduce of d_partial
 * does that).  n_peers <= 8.
 */
SPMV_B200_API int spmv_b200_pr_step_p2p(spmv_b200_pr_plan* plan, const float* d_r_old, float* d_r_new,
                                        float damping, const float* d_dsum, const uint32_t* d_bits,
                                        double* d_partial, float* const* peer_r_new, int n_peers,
                                        int self_rank, void* stream);

/*
 * The same fused exchange through NVSwitch multicast (NVLS): mc_r_new is the MULTICAST address of
 * the r_new buffers of all n_peers ranks (every rank's buffer bound at the same offset of one
 * multicast object, e.g. torch.distributed._symmetric_memory's multicast_ptr); each finished rank
 * value is sent ONCE (multimem.st) and the switch delivers it to every GPU, so a rank's NVLink
 * egress is 4 bytes per owned row instead of 4 * (n_peers - 1).  d_r_new is this rank's own
 * (unicast) mapping of its buffer.  Ordering rule as for spmv_b200_pr_step_p2p.
 */
SPMV_B200_API int spmv_b200_pr_step_multicast(spmv_b200_pr_plan* plan, const float* d_r_old,
                                              float* d_r_new, float damping, const float* d_dsum,
                                              const uint32_t* d_bits, double* d_partial,
                                              float* mc_r_new, int n_peers, int self_rank, void* stream);

/* Device buffers that other processes of the box can map (CUDA IPC): alloc returns the device
 * pointer and a 64-byte handle to send to the peers; open maps a peer's handle. */
SPMV_B200_API int spmv_b200_ipc_alloc(size_t bytes, void** d_ptr, unsigned char handle[64]);
SPMV_B200_API int spmv_b200_ipc_open(const unsigned char handle[64], void** d_ptr);
SPMV_B200_API int spmv_b200_ipc_close(void* d_ptr);
SPMV_B200_API int spmv_b200_ipc_free(void* d_ptr);

/* d_out[i] = d_r[i] / (float)sum(d_r) over n elements (f64 sum) */
SPMV_B200_API int spmv_b200_pr_normalize(const float* d_r, int n, float* d_out, void* stream);

/* whole loop on one GPU, ranks stay on the device (d_ranks [n]); the stop
 * rule and result fields are those of pagerank() (src/pagerank.cu:93-150);
 * l1_residual (optional) receives sum |r_new - r_old| of the last iteration */
SPMV_B200_API int spmv_b200_pagerank_device(const spmv_b200_csr* adj,
                                            const spmv_b200_pagerank_config* config,
                                            float* d_ranks, int* iterations,
                                            float* final_residual, bool* converged,
                                            double* l1_residual);

/* the same loop, also reporting the residual of every iteration (SURVEY 8f rank 4): l2_history[i]
 * (host array of history_capacity floats) receives the L2 norm of the delta after iteration i + 1,
 * i.e. the quantity the stop rule compares with the tolerance (src/pagerank.cu:118-127);
 * entries beyond *iterations are left untouched. */
SPMV_B200_API int spmv_b200_pagerank_device_history(const spmv_b200_csr* adj,
                                                    const spmv_b200_pagerank_config* config,
                                                    float* d_ranks, int* iterations,
                                                    float* final_residual, bool* converged,
                                                    float* l2_history, int history_capacity);

/* ---- personalized PageRank ---------------------------------------------------
 * Teleport, and the redistribution of dangling mass, follow a caller-given non-negative vector
 * `personalization` (HOST array of num_rows floats) instead of the uniform 1/n: seed-set /
 * single-source PPR, topic-sensitive or trust-biased ranking.  With v = personalization / sum(v)
 * (f64 sum in index order, each entry rounded to fp32) one iteration is
 *     r_new[i] = (d * (A r_old)[i] + (d * D) * v[i]) + (1 - d) * v[i]
 * D = dangling mass of r_old; every operation rounded separately in fp32.  r_0 = 1/n, the stop
 * rule, the residuals and the final normalisation are those of the global form.
 * INVALID_ARGUMENT, before any device work, when an entry is NaN, +-Inf or negative, when the
 * entries sum to 0, or when adj is NULL.  personalization == NULL: global PageRank (the
 * uniform vector gives the same ranks to within rounding, not bit for bit). */
/* as spmv_b200_pagerank: host ranks in out->ranks, release with spmv_b200_pagerank_free */
SPMV_B200_API int spmv_b200_pagerank_personalized(const spmv_b200_csr* adj,
                                                  const spmv_b200_pagerank_config* config,
                                                  const float* personalization,
                                                  spmv_b200_pagerank_result* out);
/* as spmv_b200_pagerank_device / _history: ranks stay on the device; l1_residual, l2_history
 * (history_capacity entries) are optional */
SPMV_B200_API int spmv_b200_pagerank_device_personalized(const spmv_b200_csr* adj,
                                                         const spmv_b200_pagerank_config* config,
                                                         const float* personalization, float* d_ranks,
                                                         int* iterations, float* final_residual,
                                                         bool* converged, double* l1_residual,
                                                         float* l2_history, int history_capacity);

/* ---- multi-GPU PageRank, host side in C++ ---------------------------------
 * The reference has no multi-GPU code.  This is the multi-GPU member of its signature family
 * pagerank(adj, config) -> ranks (reference include/spmv/pagerank.h:29-32, src/pagerank.cu:50-153):
 * contiguous row shards over the <= 8 GPUs of one NVSwitch box, every rank holding the full rank
 * vector.  Per iteration and rank: a 1-warp gate (waits for the peers' flags, folds the ranks'
 * partial sums in rank order), the fused step kernel (which also stores every finished rank value
 * into every GPU's vector: one multimem.st through the NVSwitch multicast mapping, or unicast peer
 * stores), a 1-warp publish (partial sums + flag to every peer) -- replayed from a CUDA graph, no
 * collective-library call and no host round trip between iterations.  The literal "NCCL all-gather
 * + all-reduce" transport is kept as SPMV_B200_EXCHANGE_NCCL (libnccl is dlopen'ed on first use).
 * All transports give bit-identical vectors. */
enum {
    SPMV_B200_EXCHANGE_AUTO = -1,      /* multicast if the box has NVLS, else peer stores, else NCCL */
    SPMV_B200_EXCHANGE_NCCL = 0,
    SPMV_B200_EXCHANGE_P2P = 1,
    SPMV_B200_EXCHANGE_MULTICAST = 2
};
typedef struct {
    int iterations;             /* as PageRankResult (reference include/spmv/pagerank.h:18-26) */
    float final_residual;
    int converged;
    double l1_residual;
    int iterations_launched;    /* includes the speculative iteration after convergence */
    double device_seconds;      /* CUDA events around the loop (max over ranks for pagerank_multi) */
    double wall_seconds;
    int exchange;               /* transport actually used (SPMV_B200_EXCHANGE_*) */
    int graph_replay;           /* 1: the iteration was replayed from a CUDA graph */
    int kernels_per_iteration;
} spmv_b200_pr_dist_result;

/* One process, n_gpus devices (devices == NULL: 0 .. n_gpus-1; an explicit list may name a device
 * more than once -- several ranks then share that GPU, which the peer-store transport supports):
 * adj is a HOST CSR (host arrays);
 * shards balance work(row) = nnz + row_weight; ranks_out is a host array of num_rows floats
 * (normalised, as pagerank()).  fixed_iterations > 0 runs exactly that many (no stop rule). */
SPMV_B200_API int spmv_b200_pagerank_multi(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                           int n_gpus, const int* devices, int exchange, int row_weight,
                                           int fixed_iterations, float* ranks_out,
                                           spmv_b200_pr_dist_result* out);
/* spmv_b200_pagerank_multi for personalized PageRank (personalization: host [num_rows], see
 * spmv_b200_pagerank_personalized; NULL: spmv_b200_pagerank_multi) */
SPMV_B200_API int spmv_b200_pagerank_multi_personalized(const spmv_b200_csr* adj,
                                                        const spmv_b200_pagerank_config* config,
                                                        const float* personalization, int n_gpus,
                                                        const int* devices, int exchange, int row_weight,
                                                        int fixed_iterations, float* ranks_out,
                                                        spmv_b200_pr_dist_result* out);

/* One process PER GPU (torchrun, mpirun, any launcher): a communicator for the set-up traffic
 * (shard bounds, NCCL id, descriptors of the symmetric allocations) over an abstract unix-domain
 * socket named after `session` (the same string on every rank, unique per job; one box only). */
typedef struct spmv_b200_comm spmv_b200_comm;
SPMV_B200_API int spmv_b200_comm_create(int rank, int world, const char* session, int timeout_s,
                                        spmv_b200_comm** out);
SPMV_B200_API void spmv_b200_comm_destroy(spmv_b200_comm* comm);
SPMV_B200_API int spmv_b200_comm_barrier(spmv_b200_comm* comm);
SPMV_B200_API int spmv_b200_comm_allgather(spmv_b200_comm* comm, const void* send, void* recv, size_t bytes);
/* every rank passes one open file descriptor and receives world new ones (SCM_RIGHTS) */
SPMV_B200_API int spmv_b200_comm_allgather_fds(spmv_b200_comm* comm, int my_fd, int* fds_out);

/* Sharded PageRank object: collective calls (every rank, same order).  shard = this rank's rows
 * [row_offset, row_offset + shard->num_rows) with global column ids, device arrays present
 * (borrowed).  The current device of the calling thread is the rank's GPU. */
typedef struct spmv_b200_pr_dist spmv_b200_pr_dist;
SPMV_B200_API int spmv_b200_pr_dist_create(spmv_b200_comm* comm, const spmv_b200_csr* shard, int row_offset,
                                           int n_global, int exchange, spmv_b200_pr_dist** out);
SPMV_B200_API int spmv_b200_pr_dist_run(spmv_b200_pr_dist* d, const spmv_b200_pagerank_config* config,
                                        int fixed_iterations, spmv_b200_pr_dist_result* out);
/* Personalized PageRank from the next run on (collective): every rank passes the FULL host vector
 * (n_global floats, the same on every rank; see spmv_b200_pagerank_personalized) and keeps the
 * normalised entries of its own rows.  NULL returns to global PageRank. */
SPMV_B200_API int spmv_b200_pr_dist_set_personalization(spmv_b200_pr_dist* d, const float* personalization);
/* device pointer to the full, normalised rank vector of the last run (identical on every rank) */
SPMV_B200_API const float* spmv_b200_pr_dist_ranks(const spmv_b200_pr_dist* d);
SPMV_B200_API int spmv_b200_pr_dist_exchange(const spmv_b200_pr_dist* d);
SPMV_B200_API int spmv_b200_pr_dist_hub_columns(const spmv_b200_pr_dist* d);
SPMV_B200_API void spmv_b200_pr_dist_destroy(spmv_b200_pr_dist* d);
SPMV_B200_API int spmv_b200_nccl_available(void);

#ifdef __cplusplus
} /* extern "C" */
#endif

#endif /* SPMV_B200_H */
