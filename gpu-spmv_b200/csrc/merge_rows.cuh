// merge_rows.cuh -- pieces shared by the two merge-path front ends
// (csr_merge_kernels.cu: one tile per CTA; csr_hot_kernels.cu: persistent CTAs
// with the hub columns of x in shared memory): the canonical diagonal search
// and the row epilogues (plain y store / fused PageRank update).
#pragma once

#include "device_utils.cuh"
#include "internal.hpp"

namespace spmv {
namespace b200 {
namespace {

constexpr int kT = kMergeThreads;
constexpr int kIPT = kMergeItemsPerThread;
constexpr int kTile = kMergeTile;

// ---------------------------------------------------------------- level 1 ----
// Canonical diagonal search: list A = row END offsets row_ptrs[1..rows], list
// B = non-zero indices 0..nnz-1; A wins ties (a row ends before the non-zero
// with the same index is consumed).
__device__ __forceinline__ int2 diagonal_search_global(int diagonal, const int* __restrict__ row_ptrs,
                                                       int rows, int nnz) {
    int lo = max(diagonal - nnz, 0);
    int hi = min(diagonal, rows);
    while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);
        if (__ldg(row_ptrs + mid + 1) <= diagonal - mid - 1) lo = mid + 1;
        else hi = mid;
    }
    return make_int2(lo, diagonal - lo);
}

// ------------------------------------------------- warp segmented scan ----
// Inclusive segmented scan of `v` over a warp; a lane with `head` starts a segment.  The head flags
// travel in ONE ballot and every lane derives from the mask how far back it may reach, so only the
// values are shuffled: 6 SHFL per warp instead of 12 (shuffles share the L1 data pipe with the x
// gathers, profiles/r1_hub_kernel.md).  Same additions in the same order as the (value, flag) form.
// f_incl: a head at or before this lane; ex_v / ex_f: the exclusive prefix (lane 0: 0 / 0).
__device__ __forceinline__ void warp_segmented_scan(float& v, bool head, int lane, int& f_incl, float& ex_v, int& ex_f) {
    const unsigned mask = __ballot_sync(0xffffffffu, head);
    const unsigned upto = mask & (0xffffffffu >> (31 - lane));  // heads in lanes 0..lane
    const int reach = upto ? 31 - __clz(upto) : 0;              // first lane of this lane's segment
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const float pv = __shfl_up_sync(0xffffffffu, v, d);
        if (lane - d >= reach) v = pv + v;
    }
    f_incl = upto ? 1 : 0;
    ex_v = __shfl_up_sync(0xffffffffu, v, 1);
    ex_f = (mask & ((1u << lane) - 1u)) ? 1 : 0;
    if (lane == 0) ex_v = 0.0f;
}

// -------------------------------------------------------------- epilogues ----

struct NoSums {
    __device__ __forceinline__ void clear() {}
};
struct RankSums {
    double l2, l1, dangling;
    __device__ __forceinline__ void clear() { l2 = 0.0; l1 = 0.0; dangling = 0.0; }
};

// y[row] = sum
struct PlainRow {
    using Sums = NoSums;
    static constexpr bool kReduces = false;
    float* y;
    __device__ __forceinline__ float prepare() const { return 0.0f; }
    __device__ __forceinline__ void finish(int row, float sum, Sums&, float) const { y[row] = sum; }
    __device__ __forceinline__ void tile_finish(int row, float sum, Sums&, float) const { y[row] = sum; }
    __device__ __forceinline__ void tile_epilogue(int, int, int, Sums&, float) const {}
    __device__ __forceinline__ void park(int row, float partial) const { y[row] = partial; }
    __device__ __forceinline__ float parked(int row) const { return y[row]; }
    __device__ __forceinline__ void publish_row(int) const {}
};

// fused PageRank update of one finished row.  TWO_PASS selects how a TILE applies it (below);
// the fix-up kernel always uses finish().
template <bool TWO_PASS>
struct PageRankRowT {
    using Sums = RankSums;
    static constexpr bool kReduces = true;
    PageRankStepArgs a;
    // the per-step context of dev::pr_row_value: d * dsum / n, or d * dsum when personalized
    __device__ __forceinline__ float prepare() const {
        return dev::pr_step_context(a.damping, *a.d_dsum, a.n_global, a.pvec);
    }
    __device__ __forceinline__ void finish(int row, float sum, Sums& s, float dangling_term) const {
        const int g = a.row_offset + row;
        const float v = dev::pr_row_value(a.damping, sum, dangling_term, a.teleport, a.pvec, row);
        a.r_new[g] = v;
        const double diff = static_cast<double>(v) - static_cast<double>(a.r_old[g]);
        s.l2 += diff * diff;
        s.l1 += fabs(diff);
        if ((a.bits[g >> 5] >> (g & 31)) & 1u) s.dangling += static_cast<double>(v);
    }
    // TWO_PASS: the consume loop only stores the raw row sum (tile_finish, no dependent loads in
    // the serial loop), and after a CTA-wide barrier the rows [row_lo, row_hi) the tile has finished
    // are updated together (tile_epilogue): coalesced, independent loads of r_old and the dangling
    // bits.  Same operations on the same values as finish() -> identical r_new.  Measured on R-MAT
    // 24: 3 % faster in the persistent hub-column kernel (4 workers per SM), 14 % SLOWER in the
    // one-tile-per-CTA kernel (8 CTAs per SM already hide finish()'s loads), hence the switch.
    // Either way the rows are then copied to the peers (fused slice exchange).
    __device__ __forceinline__ void tile_finish(int row, float sum, Sums& s, float dangling_term) const {
        if (TWO_PASS) a.r_new[a.row_offset + row] = sum;
        else finish(row, sum, s, dangling_term);
    }
    __device__ __forceinline__ void tile_epilogue(int row_lo, int row_hi, int tid, Sums& s, float dangling_term) const {
        const int g0 = a.row_offset + row_lo, g1 = a.row_offset + row_hi;
        if (!TWO_PASS) {
            if (a.n_peers <= 1) return;
            const volatile float* src = a.r_new;
            if (a.mc_r_new) {  // NVSwitch multicast: one store reaches every peer
                for (int g = g0 + tid; g < g1; g += kT) dev::st_multicast_f(a.mc_r_new + g, src[g]);
                return;
            }
#pragma unroll
            for (int p = 0; p < kMaxPeers; ++p) {  // static indices: the pointer table stays in the constant bank
                if (p >= a.n_peers || p == a.self_rank) continue;
                float* dst = a.peers[p];
                for (int g = g0 + tid; g < g1; g += kT) dst[g] = src[g];
            }
            return;
        }
        volatile float* mine = a.r_new;
        for (int g = g0 + tid; g < g1; g += kT) {
            const float v = dev::pr_row_value(a.damping, mine[g], dangling_term, a.teleport, a.pvec, g - a.row_offset);
            mine[g] = v;
            const double diff = static_cast<double>(v) - static_cast<double>(a.r_old[g]);
            s.l2 += diff * diff;
            s.l1 += fabs(diff);
            if ((a.bits[g >> 5] >> (g & 31)) & 1u) s.dangling += static_cast<double>(v);
            if (a.n_peers > 1) {
                if (a.mc_r_new) {
                    dev::st_multicast_f(a.mc_r_new + g, v);  // NVSwitch multicast: one store reaches every peer
                } else {
#pragma unroll
                    for (int p = 0; p < kMaxPeers; ++p)  // static indices: the pointer table stays in the constant bank
                        if (p < a.n_peers && p != a.self_rank) a.peers[p][g] = v;
                }
            }
        }
    }
    __device__ __forceinline__ void park(int row, float partial) const { a.r_new[a.row_offset + row] = partial; }
    __device__ __forceinline__ float parked(int row) const { return a.r_new[a.row_offset + row]; }
    // Fused slice exchange (the "all-gather" of the sharded iteration): tile_epilogue stores every
    // finished rank value into the r_new buffer of every peer GPU with coalesced stores over NVLink
    // -- one contiguous run per tile and peer instead of one 4-byte packet per row.
    __device__ __forceinline__ void publish_row(int row) const {  // a single row finished by the fix-up
        if (a.n_peers <= 1) return;
        const int g = a.row_offset + row;
        const float v = a.r_new[g];
        if (a.mc_r_new) {
            dev::st_multicast_f(a.mc_r_new + g, v);
            return;
        }
#pragma unroll
        for (int p = 0; p < kMaxPeers; ++p)
            if (p < a.n_peers && p != a.self_rank) a.peers[p][g] = v;
    }
};

using PageRankRow = PageRankRowT<false>;

}  // namespace
}  // namespace b200
}  // namespace spmv
