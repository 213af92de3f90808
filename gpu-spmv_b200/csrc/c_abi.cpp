// c_abi.cpp -- the extern "C" boundary declared in include/spmv_b200.h.
// Thin, exception-safe adapters over the C++ surface: the C structs are
// layout-identical to the C++ ones (asserted below), by-value results become
// out-parameters, and anything thrown is turned into a status code.
#include "spmv_b200.h"

#include "internal.hpp"
#include "pagerank_dist.hpp"

#include <cstdio>
#include <cstring>
#include <string>
#include <new>

using namespace spmv;

// ---- layout identity between the two surfaces ---------------------------------
static_assert(sizeof(spmv_b200_csr) == sizeof(CSRMatrix) && offsetof(spmv_b200_csr, d_row_ptrs) == offsetof(CSRMatrix, d_row_ptrs) &&
              offsetof(spmv_b200_csr, owns_device_memory) == offsetof(CSRMatrix, owns_device_memory), "csr");
static_assert(sizeof(spmv_b200_ell) == sizeof(ELLMatrix) && offsetof(spmv_b200_ell, d_col_indices) == offsetof(ELLMatrix, d_col_indices) &&
              offsetof(spmv_b200_ell, owns_device_memory) == offsetof(ELLMatrix, owns_device_memory), "ell");
static_assert(sizeof(spmv_b200_config) == sizeof(SpMVConfig) && offsetof(spmv_b200_config, use_texture) == offsetof(SpMVConfig, use_texture), "config");
static_assert(sizeof(spmv_b200_result) == sizeof(SpMVResult) && offsetof(spmv_b200_result, error_code) == offsetof(SpMVResult, error_code), "result");
static_assert(sizeof(spmv_b200_csr_stats) == sizeof(CSRStats), "stats");
static_assert(sizeof(spmv_b200_bandwidth) == sizeof(BandwidthMetrics), "bandwidth");
static_assert(sizeof(spmv_b200_pagerank_config) == sizeof(PageRankConfig), "pagerank config");
static_assert(sizeof(spmv_b200_pagerank_result) == sizeof(PageRankResult) && offsetof(spmv_b200_pagerank_result, converged) == offsetof(PageRankResult, converged), "pagerank result");
static_assert(sizeof(spmv_b200_topk_node) == sizeof(TopKNode), "topk");
static_assert(sizeof(spmv_b200_bench_config) == sizeof(BenchmarkConfig), "bench config");

namespace {

inline CSRMatrix* cpp(spmv_b200_csr* m) { return reinterpret_cast<CSRMatrix*>(m); }
inline const CSRMatrix* cpp(const spmv_b200_csr* m) { return reinterpret_cast<const CSRMatrix*>(m); }
inline ELLMatrix* cpp(spmv_b200_ell* m) { return reinterpret_cast<ELLMatrix*>(m); }
inline const ELLMatrix* cpp(const spmv_b200_ell* m) { return reinterpret_cast<const ELLMatrix*>(m); }
inline const SpMVConfig* cpp(const spmv_b200_config* c) { return reinterpret_cast<const SpMVConfig*>(c); }
inline const PageRankConfig* cpp(const spmv_b200_pagerank_config* c) { return reinterpret_cast<const PageRankConfig*>(c); }
inline const BenchmarkConfig* cpp(const spmv_b200_bench_config* c) { return reinterpret_cast<const BenchmarkConfig*>(c); }

constexpr int kBadArg = SPMV_B200_INVALID_ARGUMENT;

int status_of(const std::exception* e) {
    if (dynamic_cast<const std::bad_alloc*>(e)) return SPMV_B200_OUT_OF_MEMORY;
    if (dynamic_cast<const CudaException*>(e)) return SPMV_B200_CUDA_MALLOC;
    return SPMV_B200_INVALID_ARGUMENT;
}

// Runs fn(), mapping exceptions to a status.
template <typename Fn>
int guarded(Fn fn) {
    try {
        return fn();
    } catch (const std::exception& e) {
        return status_of(&e);
    } catch (...) {
        return SPMV_B200_INVALID_ARGUMENT;
    }
}

void to_c(const SpMVResult& r, spmv_b200_result* out) {
    if (!out) return;
    out->y = r.y;
    out->elapsed_ms = r.elapsed_ms;
    out->gflops = r.gflops;
    out->bandwidth_gb_s = r.bandwidth_gb_s;
    out->error_code = r.error_code;
}

void to_c(const BenchmarkResult& r, spmv_b200_bench_result* out) {
    if (!out) return;
    std::memset(out, 0, sizeof(*out));
    std::strncpy(out->name, r.name.c_str(), sizeof(out->name) - 1);
    out->execution_time_ms = r.execution_time_ms;
    out->gflops = r.gflops;
    out->bandwidth_gb_s = r.bandwidth_gb_s;
    out->avg_time_ms = r.avg_time_ms;
    out->min_time_ms = r.min_time_ms;
    out->max_time_ms = r.max_time_ms;
    out->stddev_time_ms = r.stddev_time_ms;
    out->num_runs = r.num_runs;
}

BenchmarkResult from_c(const spmv_b200_bench_result* in) {
    BenchmarkResult r;
    r.name.assign(in->name, strnlen(in->name, sizeof(in->name)));
    r.execution_time_ms = in->execution_time_ms;
    r.gflops = in->gflops;
    r.bandwidth_gb_s = in->bandwidth_gb_s;
    r.avg_time_ms = in->avg_time_ms;
    r.min_time_ms = in->min_time_ms;
    r.max_time_ms = in->max_time_ms;
    r.stddev_time_ms = in->stddev_time_ms;
    r.num_runs = in->num_runs;
    return r;
}

void to_c(const BandwidthMetrics& m, spmv_b200_bandwidth* out) {
    out->theoretical_bandwidth_gb_s = m.theoretical_bandwidth_gb_s;
    out->achieved_bandwidth_gb_s = m.achieved_bandwidth_gb_s;
    out->efficiency = m.efficiency;
}

void to_c(const SpMVConfig& c, spmv_b200_config* out) {
    out->kernel_type = static_cast<int>(c.kernel_type);
    out->block_size = c.block_size;
    out->use_texture = c.use_texture;
}

}  // namespace

extern "C" {

const char* spmv_b200_error_string(int status) { return spmv_error_string(static_cast<SpMVError>(status)); }
const char* spmv_b200_version(void) { return "spmv_b200 0.1 (sm_100a)"; }
unsigned long long spmv_b200_launch_count(void) { return b200::launch_count(); }

// ---- A. CSR ---------------------------------------------------------------------
spmv_b200_csr* spmv_b200_csr_create(int rows, int cols, int nnz) {
    try { return reinterpret_cast<spmv_b200_csr*>(csr_create(rows, cols, nnz)); } catch (...) { return nullptr; }
}
void spmv_b200_csr_destroy(spmv_b200_csr* m) { csr_destroy(cpp(m)); }
int spmv_b200_csr_from_dense(spmv_b200_csr* m, const float* dense, int rows, int cols) {
    return guarded([&] { return csr_from_dense(cpp(m), dense, rows, cols); });
}
int spmv_b200_csr_to_dense(const spmv_b200_csr* m, float* dense) { return guarded([&] { return csr_to_dense(cpp(m), dense); }); }
float spmv_b200_csr_get_element(const spmv_b200_csr* m, int row, int col) { return csr_get_element(cpp(m), row, col); }
int spmv_b200_csr_to_gpu(spmv_b200_csr* m) { return guarded([&] { return csr_to_gpu(cpp(m)); }); }
int spmv_b200_csr_from_gpu(spmv_b200_csr* m) { return guarded([&] { return csr_from_gpu(cpp(m)); }); }
void spmv_b200_csr_free_gpu(spmv_b200_csr* m) { csr_free_gpu(cpp(m)); }
int spmv_b200_csr_serialize(const spmv_b200_csr* m, const char* f) { return guarded([&] { return csr_serialize(cpp(m), f); }); }
int spmv_b200_csr_deserialize(spmv_b200_csr* m, const char* f) { return guarded([&] { return csr_deserialize(cpp(m), f); }); }
int spmv_b200_csr_compute_stats(const spmv_b200_csr* m, spmv_b200_csr_stats* out) {
    if (!out) return kBadArg;
    const CSRStats s = csr_compute_stats(cpp(m));
    out->avg_nnz_per_row = s.avg_nnz_per_row;
    out->max_nnz_per_row = s.max_nnz_per_row;
    out->min_nnz_per_row = s.min_nnz_per_row;
    out->skewness = s.skewness;
    return 0;
}

// ---- B. ELL ---------------------------------------------------------------------
spmv_b200_ell* spmv_b200_ell_create(int rows, int cols, int width) {
    try { return reinterpret_cast<spmv_b200_ell*>(ell_create(rows, cols, width)); } catch (...) { return nullptr; }
}
void spmv_b200_ell_destroy(spmv_b200_ell* m) { ell_destroy(cpp(m)); }
int spmv_b200_ell_from_dense(spmv_b200_ell* m, const float* dense, int rows, int cols) {
    return guarded([&] { return ell_from_dense(cpp(m), dense, rows, cols); });
}
int spmv_b200_ell_from_csr(spmv_b200_ell* m, const spmv_b200_csr* csr) { return guarded([&] { return ell_from_csr(cpp(m), cpp(csr)); }); }
int spmv_b200_ell_to_dense(const spmv_b200_ell* m, float* dense) { return guarded([&] { return ell_to_dense(cpp(m), dense); }); }
float spmv_b200_ell_get_element(const spmv_b200_ell* m, int row, int col) { return ell_get_element(cpp(m), row, col); }
int spmv_b200_ell_to_gpu(spmv_b200_ell* m) { return guarded([&] { return ell_to_gpu(cpp(m)); }); }
int spmv_b200_ell_from_gpu(spmv_b200_ell* m) { return guarded([&] { return ell_from_gpu(cpp(m)); }); }
void spmv_b200_ell_free_gpu(spmv_b200_ell* m) { ell_free_gpu(cpp(m)); }
int spmv_b200_ell_serialize(const spmv_b200_ell* m, const char* f) { return guarded([&] { return ell_serialize(cpp(m), f); }); }
int spmv_b200_ell_deserialize(spmv_b200_ell* m, const char* f) { return guarded([&] { return ell_deserialize(cpp(m), f); }); }
int spmv_b200_ell_index(int row, int k, int num_rows) { return ell_index(row, k, num_rows); }

// ---- C. SpMV ----------------------------------------------------------------------
void spmv_b200_spmv_cpu_csr(const spmv_b200_csr* A, const float* x, float* y) { spmv_cpu_csr(cpp(A), x, y); }
void spmv_b200_spmv_cpu_ell(const spmv_b200_ell* A, const float* x, float* y) { spmv_cpu_ell(cpp(A), x, y); }

int spmv_b200_spmv_csr(const spmv_b200_csr* A, const float* d_x, float* d_y, const spmv_b200_config* config,
                       int vec_size, spmv_b200_result* out) {
    return guarded([&] {
        const SpMVResult r = spmv_csr(cpp(A), d_x, d_y, cpp(config), vec_size);
        to_c(r, out);
        return r.error_code;
    });
}
int spmv_b200_spmv_ell(const spmv_b200_ell* A, const float* d_x, float* d_y, const spmv_b200_config* config,
                       int vec_size, spmv_b200_result* out) {
    return guarded([&] {
        const SpMVResult r = spmv_ell(cpp(A), d_x, d_y, cpp(config), vec_size);
        to_c(r, out);
        return r.error_code;
    });
}
int spmv_b200_auto_config(const spmv_b200_csr* A, spmv_b200_config* out) {
    if (!A || !out) return kBadArg;  // the C++ call dereferences A unchecked, as the reference does
    to_c(spmv_auto_config(cpp(A)), out);
    return 0;
}
int spmv_b200_reference_policy(const spmv_b200_csr* A, spmv_b200_config* out) {
    if (!A || !out) return kBadArg;
    to_c(b200::reference_policy(cpp(A)), out);
    return 0;
}
bool spmv_b200_validate_dimensions(int num_cols, int vec_size) { return spmv_validate_dimensions(num_cols, vec_size); }

int spmv_b200_spmv_csr_async(const spmv_b200_csr* A, const float* d_x, float* d_y, const spmv_b200_config* config,
                             void* stream) {
    return guarded([&] { return b200::spmv_csr_async(cpp(A), d_x, d_y, cpp(config), static_cast<cudaStream_t>(stream)); });
}
int spmv_b200_spmv_ell_async(const spmv_b200_ell* A, const float* d_x, float* d_y, void* stream) {
    return guarded([&] { return b200::spmv_ell_async(cpp(A), d_x, d_y, static_cast<cudaStream_t>(stream)); });
}

int spmv_b200_ell_host_plan_create(const spmv_b200_ell* A, int chunks, spmv_b200_ell_host_plan** out) {
    return guarded([&] { return b200::ell_host_plan_create(cpp(A), chunks, reinterpret_cast<b200::EllHostPlan**>(out)); });
}
void spmv_b200_ell_host_plan_destroy(spmv_b200_ell_host_plan* plan) {
    b200::ell_host_plan_destroy(reinterpret_cast<b200::EllHostPlan*>(plan));
}
int spmv_b200_spmv_ell_host(spmv_b200_ell_host_plan* plan, const float* x_host, float* y_host) {
    return guarded([&] { return b200::spmv_ell_host(reinterpret_cast<b200::EllHostPlan*>(plan), x_host, y_host); });
}
int spmv_b200_ell_host_plan_info(const spmv_b200_ell_host_plan* plan, int* chunks, int* ranged, int* max_lookahead) {
    if (!plan) return kBadArg;
    b200::ell_host_plan_info(reinterpret_cast<const b200::EllHostPlan*>(plan), chunks, ranged, max_lookahead);
    return 0;
}

int spmv_b200_ell_host_plan_bytes(const spmv_b200_ell_host_plan* plan, unsigned long long* h2d, unsigned long long* d2h) {
    if (!plan) return kBadArg;
    b200::ell_host_plan_bytes(reinterpret_cast<const b200::EllHostPlan*>(plan), h2d, d2h);
    return 0;
}

int spmv_b200_ell_host_plan_gated(const spmv_b200_ell_host_plan* plan, int* gated, int* x_chunks) {
    if (!plan) return kBadArg;
    b200::ell_host_plan_gated(reinterpret_cast<const b200::EllHostPlan*>(plan), gated, x_chunks);
    return 0;
}

int spmv_b200_probe_h2d_order(const float* x_host, unsigned long long n, int samples, long long* out_ns, int mode, unsigned sleep_ns) {
    return guarded([&] { return b200::probe_h2d_order(x_host, static_cast<size_t>(n), samples, out_ns, mode, sleep_ns); });
}

// ---- D. bandwidth / PageRank / benchmark ------------------------------------------------
int spmv_b200_bandwidth_csr(const spmv_b200_csr* A, float ms, spmv_b200_bandwidth* out) {
    if (!out) return kBadArg;
    to_c(compute_bandwidth_csr(cpp(A), ms), out);
    return 0;
}
int spmv_b200_bandwidth_ell(const spmv_b200_ell* A, float ms, spmv_b200_bandwidth* out) {
    if (!out) return kBadArg;
    to_c(compute_bandwidth_ell(cpp(A), ms), out);
    return 0;
}
float spmv_b200_peak_bandwidth(void) { return get_gpu_peak_bandwidth(); }

int spmv_b200_pagerank(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                       spmv_b200_pagerank_result* out) {
    if (!out) return kBadArg;
    return guarded([&] {
        const PageRankResult r = pagerank(cpp(adj), cpp(config));
        out->ranks = r.ranks;
        out->iterations = r.iterations;
        out->final_residual = r.final_residual;
        out->converged = r.converged;
        return 0;
    });
}
int spmv_b200_pagerank_personalized(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                    const float* personalization, spmv_b200_pagerank_result* out) {
    if (!adj || !out) return kBadArg;
    return guarded([&] {
        PageRankResult r;
        const int rc = b200::pagerank_to_host(cpp(adj), cpp(config), personalization, &r);
        out->ranks = r.ranks;
        out->iterations = r.iterations;
        out->final_residual = r.final_residual;
        out->converged = r.converged;
        return rc;
    });
}
void spmv_b200_pagerank_free(spmv_b200_pagerank_result* r) { pagerank_free(reinterpret_cast<PageRankResult*>(r)); }
int spmv_b200_pagerank_top_k(const spmv_b200_pagerank_result* r, int num_nodes, int k, spmv_b200_topk_node* top_k) {
    if (!r || !r->ranks || !top_k || k <= 0) return kBadArg;
    return guarded([&] {
        pagerank_top_k(reinterpret_cast<const PageRankResult*>(r), num_nodes, k, reinterpret_cast<TopKNode*>(top_k));
        return 0;
    });
}

int spmv_b200_benchmark_csr(const spmv_b200_csr* A, const float* x, const spmv_b200_config* config,
                            const spmv_b200_bench_config* bc, spmv_b200_bench_result* out) {
    if (!A || !x || !out) return kBadArg;
    return guarded([&] {
        to_c(benchmark_csr(cpp(A), x, cpp(config), cpp(bc)), out);
        return 0;
    });
}
int spmv_b200_benchmark_ell(const spmv_b200_ell* A, const float* x, const spmv_b200_bench_config* bc,
                            spmv_b200_bench_result* out) {
    if (!A || !x || !out) return kBadArg;
    return guarded([&] {
        to_c(benchmark_ell(cpp(A), x, cpp(bc)), out);
        return 0;
    });
}
int spmv_b200_compare_gpu_cpu_csr(const spmv_b200_csr* A, const float* x, const spmv_b200_config* config,
                                  const spmv_b200_bench_config* bc, spmv_b200_bench_result* gpu_out,
                                  spmv_b200_bench_result* cpu_out, float* speedup) {
    if (!A || !x) return kBadArg;
    return guarded([&] {
        const ComparisonResult c = compare_gpu_cpu_csr(cpp(A), x, cpp(config), cpp(bc));
        to_c(c.gpu_result, gpu_out);
        to_c(c.cpu_result, cpu_out);
        if (speedup) *speedup = c.speedup;
        return 0;
    });
}
int spmv_b200_benchmark_to_json(const spmv_b200_bench_result* r, char* buf, int cap) {
    if (!r || !buf || cap <= 0) return -1;
    try {
        const std::string s = benchmark_to_json(from_c(r));
        if (static_cast<int>(s.size()) + 1 > cap) return -1;
        std::memcpy(buf, s.c_str(), s.size() + 1);
        return static_cast<int>(s.size());
    } catch (...) {
        return -1;
    }
}
int spmv_b200_benchmark_from_json(const char* json, spmv_b200_bench_result* out) {
    if (!json || !out) return kBadArg;
    return guarded([&] {
        to_c(benchmark_from_json(json), out);
        return 0;
    });
}

int spmv_b200_benchmark_csr_report(const spmv_b200_csr* A_c, const float* x, const spmv_b200_config* config,
                                   const spmv_b200_bench_config* bench_config, float peak_gb_s, char* buf, int cap) {
    const CSRMatrix* A = cpp(A_c);
    if (!A || !x || !buf || cap <= 0) return kBadArg;
    if (!A->d_row_ptrs || (A->nnz > 0 && (!A->d_col_indices || !A->d_values))) return SPMV_B200_INVALID_FORMAT;
    int rc = -1;
    const int status = guarded([&] {
        SpMVConfig chosen = config ? *cpp(config) : spmv_auto_config(A);
        const BenchmarkConfig defaults;
        const BenchmarkConfig& bc = bench_config ? *cpp(bench_config) : defaults;
        BenchmarkResult gpu;
        float cpu_ms = 0.0f, speedup = 0.0f;
        if (bc.compare_cpu && A->row_ptrs && (A->nnz == 0 || (A->values && A->col_indices))) {
            const ComparisonResult cmp = compare_gpu_cpu_csr(A, x, &chosen, &bc);
            gpu = cmp.gpu_result;
            cpu_ms = cmp.cpu_result.avg_time_ms;
            speedup = cmp.speedup;
        } else {
            gpu = benchmark_csr(A, x, &chosen, &bc);
        }
        const double bytes = static_cast<double>(b200::csr_compulsory_bytes(A));
        const double peak = peak_gb_s > 0.0f ? peak_gb_s : get_gpu_peak_bandwidth();
        const double eff = gpu.avg_time_ms > 0.0f ? bytes / 1e9 / (gpu.avg_time_ms * 1e-3) : 0.0;
        static const char* names[] = {"SCALAR_CSR", "VECTOR_CSR", "MERGE_PATH", "ELL_KERNEL"};
        const int k = static_cast<int>(chosen.kernel_type);
        std::string js = benchmark_to_json(gpu);
        js.erase(js.size() - 2);  // drop the closing "\n}" and append the roofline figures
        char extra[640];
        std::snprintf(extra, sizeof extra,
                      ",\n  \"kernel\": \"%s\",\n  \"algorithmic_bytes\": %.0f,\n  \"effective_gb_s\": %.6f,\n"
                      "  \"peak_gb_s\": %.6f,\n  \"roofline_fraction\": %.6f,\n  \"cpu_avg_time_ms\": %.6f,\n"
                      "  \"cpu_threads\": %d,\n  \"speedup\": %.6f\n}",
                      (k >= 0 && k < 4) ? names[k] : "SCALAR_CSR", bytes, eff, peak, peak > 0.0 ? eff / peak : 0.0,
                      static_cast<double>(cpu_ms), cpu_ms > 0.0f ? 1 : 0, static_cast<double>(speedup));
        js += extra;
        if (static_cast<int>(js.size()) + 1 > cap) return 0;  // rc stays -1
        std::memcpy(buf, js.c_str(), js.size() + 1);
        rc = static_cast<int>(js.size());
        return 0;
    });
    return status != 0 ? status : rc;
}

int spmv_b200_set_l2_fetch_granularity(int bytes) {
    if (bytes != 32 && bytes != 64 && bytes != 128) return kBadArg;
    if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, static_cast<size_t>(bytes)) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_KERNEL_LAUNCH;
    }
    return 0;
}
int spmv_b200_l2_persistence_limits(unsigned long long* max_set_aside_bytes, unsigned long long* max_window_bytes, unsigned long long* l2_bytes) {
    int dev = 0, a = 0, b = 0, c = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&a, cudaDevAttrMaxPersistingL2CacheSize, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&b, cudaDevAttrMaxAccessPolicyWindowSize, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&c, cudaDevAttrL2CacheSize, dev) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_KERNEL_LAUNCH;
    }
    if (max_set_aside_bytes) *max_set_aside_bytes = static_cast<unsigned long long>(a);
    if (max_window_bytes) *max_window_bytes = static_cast<unsigned long long>(b);
    if (l2_bytes) *l2_bytes = static_cast<unsigned long long>(c);
    return 0;
}
int spmv_b200_set_l2_persistence(void* stream, const void* base, unsigned long long bytes, float hit_ratio, unsigned long long set_aside_bytes) {
    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, static_cast<size_t>(set_aside_bytes)) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_KERNEL_LAUNCH;
    }
    cudaStreamAttrValue v;
    std::memset(&v, 0, sizeof(v));
    v.accessPolicyWindow.base_ptr = const_cast<void*>(base);
    v.accessPolicyWindow.num_bytes = base ? static_cast<size_t>(bytes) : 0;
    v.accessPolicyWindow.hitRatio = hit_ratio;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(static_cast<cudaStream_t>(stream), cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_KERNEL_LAUNCH;
    }
    if (!base) cudaCtxResetPersistingL2Cache();
    return 0;
}
int spmv_b200_get_l2_fetch_granularity(void) {
    size_t v = 0;
    if (cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_KERNEL_LAUNCH;
    }
    return static_cast<int>(v);
}

// ---- E. extensions ----------------------------------------------------------------------

int spmv_b200_ell_from_csr_device(spmv_b200_ell* ell_c, const spmv_b200_csr* csr_c) {
    ELLMatrix* ell = cpp(ell_c);
    const CSRMatrix* csr = cpp(csr_c);
    if (!ell || !csr) return kBadArg;
    if (!csr->d_row_ptrs || (csr->nnz > 0 && (!csr->d_col_indices || !csr->d_values))) return SPMV_B200_INVALID_FORMAT;
    return guarded([&] {
        ell_free_gpu(ell);
        const b200::CsrView A = b200::view_of(csr);
        int width = 0;
        if (A.rows > 0) {
            int* d_w = nullptr;
            CUDA_CHECK(cudaMalloc(&d_w, sizeof(int)));
            cudaMemset(d_w, 0, sizeof(int));
            b200::launch_max_row_len(A, d_w, nullptr);
            cudaError_t e = cudaMemcpy(&width, d_w, sizeof(int), cudaMemcpyDeviceToHost);
            cudaFree(d_w);
            if (e != cudaSuccess) return static_cast<int>(SPMV_B200_CUDA_MEMCPY);
        }
        ell->num_rows = csr->num_rows;
        ell->num_cols = csr->num_cols;
        ell->max_nnz_per_row = width;
        const size_t slots = static_cast<size_t>(A.rows > 0 ? A.rows : 0) * width;
        if (slots) {
            CUDA_CHECK(cudaMalloc(&ell->d_values, slots * sizeof(float)));
            CUDA_CHECK(cudaMalloc(&ell->d_col_indices, slots * sizeof(int)));
            if (b200::launch_ell_from_csr(A, width, ell->d_values, ell->d_col_indices, nullptr) != cudaSuccess)
                return static_cast<int>(SPMV_B200_KERNEL_LAUNCH);
            CUDA_CHECK(cudaDeviceSynchronize());
        }
        ell->owns_device_memory = true;
        return 0;
    });
}

int spmv_b200_merge_path_search(int diagonal, const int* row_ptrs, int num_rows, int nnz, int* out_row, int* out_nz) {
    if (!row_ptrs || !out_row || !out_nz || diagonal < 0 || static_cast<long long>(diagonal) > static_cast<long long>(num_rows) + nnz)
        return kBadArg;
    int lo = diagonal - nnz > 0 ? diagonal - nnz : 0;
    int hi = diagonal < num_rows ? diagonal : num_rows;
    while (lo < hi) {  // same predicate as diagonal_search_global in csr_merge_kernels.cu
        const int mid = lo + ((hi - lo) >> 1);
        if (row_ptrs[mid + 1] <= diagonal - mid - 1) lo = mid + 1;
        else hi = mid;
    }
    *out_row = lo;
    *out_nz = diagonal - lo;
    return 0;
}

// Contiguous row split balancing work(row) = nnz(row) + row_weight: bounds[p] = first row whose
// prefix work (row_ptrs[i] + i * row_weight) is >= p * total / parts.
int spmv_b200_partition_rows_weighted(const int* row_ptrs, int num_rows, int parts, int row_weight, int* bounds) {
    if (!row_ptrs || !bounds || num_rows < 0 || parts <= 0 || row_weight < 0) return kBadArg;
    const long long total = static_cast<long long>(row_ptrs[num_rows]) + static_cast<long long>(num_rows) * row_weight;
    bounds[0] = 0;
    for (int p = 1; p < parts; ++p) {
        const long long target = total * p / parts;
        int lo = 0, hi = num_rows;
        while (lo < hi) {
            const int mid = lo + ((hi - lo) >> 1);
            if (row_ptrs[mid] + static_cast<long long>(mid) * row_weight < target) lo = mid + 1;
            else hi = mid;
        }
        bounds[p] = lo < bounds[p - 1] ? bounds[p - 1] : lo;
    }
    bounds[parts] = num_rows;
    return 0;
}

// nnz-balanced split (row_weight 0)
int spmv_b200_partition_rows(const int* row_ptrs, int num_rows, int parts, int* bounds) {
    return spmv_b200_partition_rows_weighted(row_ptrs, num_rows, parts, 0, bounds);
}

int spmv_b200_pagerank_top_k_device(const float* d_ranks, int num_nodes, int k, spmv_b200_topk_node* top_k) {
    return guarded([&] {
        return b200::pagerank_top_k_device(d_ranks, num_nodes, k, reinterpret_cast<TopKNode*>(top_k));
    });
}

int spmv_b200_csr_load_matrix_market(spmv_b200_csr* out, const char* filename) {
    return guarded([&] { return b200::csr_load_matrix_market(cpp(out), filename); });
}
int spmv_b200_csr_save_matrix_market(const spmv_b200_csr* m, const char* filename) {
    return guarded([&] { return b200::csr_save_matrix_market(cpp(m), filename); });
}

int spmv_b200_csr_from_coo_device(spmv_b200_csr* out, int rows, int cols, long long n_entries, const int* d_row_indices,
                                  const int* d_col_indices, const float* d_values) {
    return guarded([&] {
        return b200::csr_from_coo_device(cpp(out), rows, cols, n_entries, d_row_indices, d_col_indices, d_values);
    });
}
int spmv_b200_csr_normalize_columns_device(spmv_b200_csr* A) {
    return guarded([&] { return b200::csr_normalize_columns_device(cpp(A)); });
}

int spmv_b200_csr_plan_create(const spmv_b200_csr* A, int max_hot_columns, int force, spmv_b200_csr_plan** out) {
    return guarded([&] {
        return b200::csr_plan_create(cpp(A), max_hot_columns, force, reinterpret_cast<b200::CsrPlan**>(out));
    });
}
void spmv_b200_csr_plan_destroy(spmv_b200_csr_plan* plan) { b200::csr_plan_destroy(reinterpret_cast<b200::CsrPlan*>(plan)); }
int spmv_b200_csr_plan_refresh_values(spmv_b200_csr_plan* plan, void* stream) {
    return guarded([&] {
        return b200::csr_plan_refresh_values(reinterpret_cast<b200::CsrPlan*>(plan), static_cast<cudaStream_t>(stream));
    });
}
int spmv_b200_csr_plan_info(const spmv_b200_csr_plan* plan, int* hot_columns, long long* hot_nnz, int* mode) {
    if (!plan) return kBadArg;
    b200::csr_plan_info(reinterpret_cast<const b200::CsrPlan*>(plan), hot_columns, hot_nnz, mode);
    return 0;
}
int spmv_b200_spmv_csr_planned(const spmv_b200_csr_plan* plan, const float* d_x, float* d_y, void* stream) {
    return guarded([&] {
        return b200::spmv_csr_planned(reinterpret_cast<const b200::CsrPlan*>(plan), d_x, d_y,
                                      static_cast<cudaStream_t>(stream));
    });
}
int spmv_b200_csr_auto_plan_info(const spmv_b200_csr* A, int* hot_columns, long long* hot_nnz) {
    if (!A) return kBadArg;
    b200::auto_plan_info(cpp(A), hot_columns, hot_nnz);
    return 0;
}
void spmv_b200_set_auto_plan(int enabled) { b200::set_auto_plan(enabled != 0); }
int spmv_b200_auto_plan_enabled(void) { return b200::auto_plan_enabled() ? 1 : 0; }
void spmv_b200_csr_forget_plan(const spmv_b200_csr* A) {
    if (A) b200::forget_device_csr(cpp(A)->d_col_indices);
}

int spmv_b200_pr_plan_set_hot(spmv_b200_pr_plan* plan, int max_hot_columns, int force, void* stream) {
    return guarded([&] {
        return b200::pr_plan_set_hot(reinterpret_cast<b200::PrPlan*>(plan), max_hot_columns, force != 0,
                                     static_cast<cudaStream_t>(stream));
    });
}

int spmv_b200_pr_plan_create(const spmv_b200_csr* shard, int row_offset, int n_global, void* stream,
                             spmv_b200_pr_plan** out) {
    return guarded([&] {
        return b200::pr_plan_create(cpp(shard), row_offset, n_global, static_cast<cudaStream_t>(stream),
                                    reinterpret_cast<b200::PrPlan**>(out));
    });
}
void spmv_b200_pr_plan_destroy(spmv_b200_pr_plan* plan) { b200::pr_plan_destroy(reinterpret_cast<b200::PrPlan*>(plan)); }

int spmv_b200_pr_colsum(const spmv_b200_pr_plan* plan, double* d_colsum, void* stream) {
    if (!plan || !d_colsum) return kBadArg;
    const cudaError_t e = b200::launch_colsum(b200::pr_plan_view(reinterpret_cast<const b200::PrPlan*>(plan)), d_colsum,
                                              static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? 0 : SPMV_B200_KERNEL_LAUNCH;
}
int spmv_b200_pr_dangling_bits(const double* d_colsum, int n, uint32_t* d_bits, void* stream) {
    if (!d_colsum || !d_bits || n < 0) return kBadArg;
    return b200::launch_dangling_bits(d_colsum, n, n, d_bits, static_cast<cudaStream_t>(stream)) == cudaSuccess
               ? 0 : SPMV_B200_KERNEL_LAUNCH;
}
int spmv_b200_pr_init(int n, const uint32_t* d_bits, float* d_r, float* d_dsum, void* stream) {
    if (!d_bits || !d_r || !d_dsum || n < 0) return kBadArg;
    return guarded([&] {
        double* tmp = nullptr;
        CUDA_CHECK(cudaMalloc(&tmp, sizeof(double) * b200::kPrScratchDoubles));
        const cudaError_t e = b200::launch_pr_init(n, d_bits, d_r, d_dsum, tmp, static_cast<cudaStream_t>(stream));
        cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
        cudaFree(tmp);
        return e == cudaSuccess ? 0 : static_cast<int>(SPMV_B200_KERNEL_LAUNCH);
    });
}
int spmv_b200_pr_step(spmv_b200_pr_plan* plan, const float* d_r_old, float* d_r_new, float damping,
                      const float* d_dsum, const uint32_t* d_bits, double* d_partial, void* stream) {
    return guarded([&] {
        return b200::pr_step(reinterpret_cast<b200::PrPlan*>(plan), d_r_old, d_r_new, damping, d_dsum, d_bits, d_partial,
                             static_cast<cudaStream_t>(stream));
    });
}
int spmv_b200_pr_step_p2p(spmv_b200_pr_plan* plan, const float* d_r_old, float* d_r_new, float damping,
                          const float* d_dsum, const uint32_t* d_bits, double* d_partial, float* const* peer_r_new,
                          int n_peers, int self_rank, void* stream) {
    return guarded([&] {
        return b200::pr_step(reinterpret_cast<b200::PrPlan*>(plan), d_r_old, d_r_new, damping, d_dsum, d_bits, d_partial,
                             static_cast<cudaStream_t>(stream), peer_r_new, n_peers, self_rank);
    });
}

int spmv_b200_pr_step_multicast(spmv_b200_pr_plan* plan, const float* d_r_old, float* d_r_new, float damping,
                                const float* d_dsum, const uint32_t* d_bits, double* d_partial, float* mc_r_new,
                                int n_peers, int self_rank, void* stream) {
    if (!mc_r_new) return kBadArg;
    return guarded([&] {
        return b200::pr_step(reinterpret_cast<b200::PrPlan*>(plan), d_r_old, d_r_new, damping, d_dsum, d_bits, d_partial,
                             static_cast<cudaStream_t>(stream), nullptr, n_peers, self_rank, mc_r_new);
    });
}

static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");

int spmv_b200_ipc_alloc(size_t bytes, void** d_ptr, unsigned char handle[64]) {
    if (!d_ptr || !handle || bytes == 0) return kBadArg;
    if (cudaMalloc(d_ptr, bytes) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_CUDA_MALLOC;
    }
    cudaIpcMemHandle_t h;
    if (cudaIpcGetMemHandle(&h, *d_ptr) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(*d_ptr);
        *d_ptr = nullptr;
        return SPMV_B200_CUDA_MALLOC;
    }
    std::memcpy(handle, &h, 64);
    return 0;
}
int spmv_b200_ipc_open(const unsigned char handle[64], void** d_ptr) {
    if (!d_ptr || !handle) return kBadArg;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    if (cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        return SPMV_B200_CUDA_MALLOC;
    }
    return 0;
}
int spmv_b200_ipc_close(void* d_ptr) { return cudaIpcCloseMemHandle(d_ptr) == cudaSuccess ? 0 : SPMV_B200_CUDA_MALLOC; }
int spmv_b200_ipc_free(void* d_ptr) { return cudaFree(d_ptr) == cudaSuccess ? 0 : SPMV_B200_CUDA_MALLOC; }

int spmv_b200_pr_normalize(const float* d_r, int n, float* d_out, void* stream) {
    if (!d_r || !d_out || n < 0) return kBadArg;
    return guarded([&] {
        double* tmp = nullptr;
        CUDA_CHECK(cudaMalloc(&tmp, sizeof(double) * b200::kPrScratchDoubles));
        const cudaError_t e = b200::launch_normalize(d_r, n, d_out, tmp, static_cast<cudaStream_t>(stream));
        cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
        cudaFree(tmp);
        return e == cudaSuccess ? 0 : static_cast<int>(SPMV_B200_KERNEL_LAUNCH);
    });
}

int spmv_b200_pagerank_device_history(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, float* d_ranks,
                                      int* iterations, float* final_residual, bool* converged, float* l2_history,
                                      int history_capacity) {
    if (history_capacity < 0 || (history_capacity > 0 && !l2_history)) return kBadArg;
    return guarded([&] {
        return b200::pagerank_device(cpp(adj), cpp(config), d_ranks, iterations, final_residual, converged, nullptr, true,
                                     l2_history, history_capacity);
    });
}

int spmv_b200_pagerank_device(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, float* d_ranks,
                              int* iterations, float* final_residual, bool* converged, double* l1_residual) {
    return guarded([&] {
        return b200::pagerank_device(cpp(adj), cpp(config), d_ranks, iterations, final_residual, converged, l1_residual);
    });
}

int spmv_b200_pagerank_device_personalized(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                           const float* personalization, float* d_ranks, int* iterations,
                                           float* final_residual, bool* converged, double* l1_residual,
                                           float* l2_history, int history_capacity) {
    if (!adj || !d_ranks || history_capacity < 0 || (history_capacity > 0 && !l2_history)) return kBadArg;
    return guarded([&] {
        float* d_pvec = nullptr;
        int rc = b200::pr_personalization_upload(personalization, cpp(adj)->num_rows, 0, cpp(adj)->num_rows, &d_pvec,
                                                  nullptr);
        if (rc != 0) return rc;
        rc = b200::pagerank_device(cpp(adj), cpp(config), d_ranks, iterations, final_residual, converged, l1_residual, true,
                                   l2_history, history_capacity, d_pvec);
        cudaFree(d_pvec);
        return rc;
    });
}

}  // extern "C"

// ---- multi-GPU PageRank ---------------------------------------------------------------------
static_assert(sizeof(spmv_b200_pr_dist_result) == sizeof(b200::PrDistResult) &&
              offsetof(spmv_b200_pr_dist_result, device_seconds) == offsetof(b200::PrDistResult, device_seconds) &&
              offsetof(spmv_b200_pr_dist_result, kernels_per_iteration) == offsetof(b200::PrDistResult, kernels_per_iteration),
              "pr_dist result");

int spmv_b200_pagerank_multi(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config, int n_gpus,
                             const int* devices, int exchange, int row_weight, int fixed_iterations, float* ranks_out,
                             spmv_b200_pr_dist_result* out) {
    return guarded([&] {
        return b200::pagerank_multi(cpp(adj), cpp(config), n_gpus, devices, exchange, row_weight, fixed_iterations,
                                    ranks_out, reinterpret_cast<b200::PrDistResult*>(out));
    });
}
int spmv_b200_pagerank_multi_personalized(const spmv_b200_csr* adj, const spmv_b200_pagerank_config* config,
                                          const float* personalization, int n_gpus, const int* devices, int exchange,
                                          int row_weight, int fixed_iterations, float* ranks_out,
                                          spmv_b200_pr_dist_result* out) {
    return guarded([&] {
        return b200::pagerank_multi(cpp(adj), cpp(config), n_gpus, devices, exchange, row_weight, fixed_iterations,
                                    ranks_out, reinterpret_cast<b200::PrDistResult*>(out), personalization);
    });
}
int spmv_b200_comm_create(int rank, int world, const char* session, int timeout_s, spmv_b200_comm** out) {
    return guarded([&] {
        b200::Comm* c = nullptr;
        if (!out || b200::comm_create_socket(rank, world, session, timeout_s, &c) != 0) return kBadArg;
        *out = reinterpret_cast<spmv_b200_comm*>(c);
        return 0;
    });
}
void spmv_b200_comm_destroy(spmv_b200_comm* comm) { delete reinterpret_cast<b200::Comm*>(comm); }
int spmv_b200_comm_barrier(spmv_b200_comm* comm) {
    return comm ? (reinterpret_cast<b200::Comm*>(comm)->barrier() == 0 ? 0 : SPMV_B200_FILE_IO) : kBadArg;
}
int spmv_b200_comm_allgather(spmv_b200_comm* comm, const void* send, void* recv, size_t bytes) {
    if (!comm || !send || !recv) return kBadArg;
    return reinterpret_cast<b200::Comm*>(comm)->allgather(send, recv, bytes) == 0 ? 0 : SPMV_B200_FILE_IO;
}
int spmv_b200_comm_allgather_fds(spmv_b200_comm* comm, int my_fd, int* fds_out) {
    if (!comm || !fds_out || my_fd < 0) return kBadArg;
    return reinterpret_cast<b200::Comm*>(comm)->allgather_fds(my_fd, fds_out) == 0 ? 0 : SPMV_B200_FILE_IO;
}
int spmv_b200_pr_dist_create(spmv_b200_comm* comm, const spmv_b200_csr* shard, int row_offset, int n_global, int exchange,
                             spmv_b200_pr_dist** out) {
    return guarded([&] {
        return b200::pr_dist_create(reinterpret_cast<b200::Comm*>(comm), cpp(shard), row_offset, n_global, exchange,
                                    reinterpret_cast<b200::PrDist**>(out));
    });
}
int spmv_b200_pr_dist_run(spmv_b200_pr_dist* d, const spmv_b200_pagerank_config* config, int fixed_iterations,
                          spmv_b200_pr_dist_result* out) {
    return guarded([&] {
        return b200::pr_dist_run(reinterpret_cast<b200::PrDist*>(d), cpp(config), fixed_iterations,
                                 reinterpret_cast<b200::PrDistResult*>(out));
    });
}
int spmv_b200_pr_dist_set_personalization(spmv_b200_pr_dist* d, const float* personalization) {
    return guarded([&] { return b200::pr_dist_set_personalization(reinterpret_cast<b200::PrDist*>(d), personalization); });
}
const float* spmv_b200_pr_dist_ranks(const spmv_b200_pr_dist* d) { return b200::pr_dist_ranks(reinterpret_cast<const b200::PrDist*>(d)); }
int spmv_b200_pr_dist_exchange(const spmv_b200_pr_dist* d) { return b200::pr_dist_exchange(reinterpret_cast<const b200::PrDist*>(d)); }
int spmv_b200_pr_dist_hub_columns(const spmv_b200_pr_dist* d) { return b200::pr_dist_hub_columns(reinterpret_cast<const b200::PrDist*>(d)); }
void spmv_b200_pr_dist_destroy(spmv_b200_pr_dist* d) { b200::pr_dist_destroy(reinterpret_cast<b200::PrDist*>(d)); }
int spmv_b200_nccl_available(void) { return b200::nccl_available() ? 1 : 0; }
