// device_utils.cuh -- sm_100a load/store, TMA (1-D bulk copy) and mbarrier
// primitives shared by the SpMV kernels.  Inline PTX only; no libraries.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace spmv {
namespace b200 {
namespace dev {

// ---- streaming loads of matrix data (read once: keep out of L1) ------------

__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ int4 ld_stream_i4(const int* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ld_stream_f2(const float* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];"
                 : "=f"(r.x), "=f"(r.y)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ int2 ld_stream_i2(const int* p) {
    int2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.s32 {%0, %1}, [%2];"
                 : "=r"(r.x), "=r"(r.y)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float ld_stream_f(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ int ld_stream_i(const int* p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// ---- L2 eviction-priority hints (createpolicy + ld ... .L2::cache_hint) ---------
// The matrix stream is read once: evict_first keeps it from pushing the re-used x entries out of L2.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float ld_stream_f_hint(const float* p, uint64_t policy) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(policy));
    return r;
}
__device__ __forceinline__ int ld_stream_i_hint(const int* p, uint64_t policy) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(policy));
    return r;
}

// ---- gathers of x (re-used: read-only path, L1-allocating) -----------------

__device__ __forceinline__ float ld_x(const float* p) {
    float r;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// ---- streaming stores of y -------------------------------------------------

__device__ __forceinline__ void st_stream_f4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream_f2(float* p, float2 v) {
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};"
                 :: "l"(p), "f"(v.x), "f"(v.y) : "memory");
}

// ---- NVSwitch multicast store (NVLS): one store, delivered to every GPU bound to the multicast
// object the address belongs to.  SASS: a store to a multicast-mapped address.
__device__ __forceinline__ void st_multicast_f(float* mc_addr, float v) {
    asm volatile("multimem.st.weak.global.f32 [%0], %1;" :: "l"(mc_addr), "f"(v) : "memory");
}

// ---- shared-memory address helper -------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D TMA bulk copy (global -> shared) -------------------------
// cp.async.bulk needs: 16-byte aligned global and shared addresses and a byte
// count that is a multiple of 16.  SASS: UBLKCP.

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t arrivals) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(arrivals));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                             uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool aligned16(const void* p) {
    return (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
}

// ---- PageRank row update ------------------------------------------------------
// The one definition of the update, used by every PageRank epilogue (PageRankRowT::finish and
// ::tile_epilogue, seg_pagerank_epilogue_kernel, pagerank_small_kernel).  pvec selects the form
// at run time; the branch is uniform over the kernel.
//   pvec == nullptr  global PageRank:      r = (d*y + d*D/n) + teleport,          teleport = (1-d)/n
//   pvec != nullptr  personalized PageRank: r = (d*y + (d*D)*v[i]) + teleport*v[i], teleport = 1-d
// D is the dangling mass of r_old and v the normalised personalization vector.  Every operation
// is rounded separately (no FMA contraction), so the global form is exactly the reference's
// expression (src/pagerank.cu:111-113, left to right in fp32).
// Per-step context: d*D/n, or d*D in the personalized form.
__device__ __forceinline__ float pr_step_context(float damping, float dsum, int n, const float* pvec) {
    const float dd = __fmul_rn(damping, dsum);
    return pvec ? dd : __fdiv_rn(dd, static_cast<float>(n));
}
// New rank of one row from its product y; local_row indexes pvec (the rows of this shard).
__device__ __forceinline__ float pr_row_value(float damping, float y, float ctx, float teleport, const float* pvec,
                                              int local_row) {
    const float dy = __fmul_rn(damping, y);
    if (!pvec) return __fadd_rn(__fadd_rn(dy, ctx), teleport);
    const float v = __ldg(pvec + local_row);
    return __fadd_rn(__fadd_rn(dy, __fmul_rn(ctx, v)), __fmul_rn(teleport, v));
}

// ---- ordering ----------------------------------------------------------------

// Order-preserving uint32 image of a float for radix selection: larger float <=> larger key (NaN sorts high);
// -0 and +0 map to the same key.
__device__ __forceinline__ unsigned order_key(float v) {
    const unsigned u = v == 0.0f ? 0u : __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---- warp reductions ---------------------------------------------------------

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ unsigned warp_sum(unsigned v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    return v;
}

}  // namespace dev
}  // namespace b200
}  // namespace spmv
