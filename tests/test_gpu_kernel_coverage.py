"""Every kernel the library ships, run and checked against the oracle -- with finite inputs and with IEEE specials.

The dispatch picks a kernel by the matrix's structure and by tuning variables (SPMV_B200_*) read once per process.
CASES below names, for each instantiation, a matrix that selects it, the variables that force it, the entry point,
the kernel names the case must launch and the rule its result is held to.  The cases of one variable set run in one
child process (this file with --child); under torch.profiler every case records the kernels it launched, and the
coverage gate asserts that observed kernels together with NOT_RUN_HERE are exactly the kernels in
libspmv_b200.so (cuobjdump, scripts/sass_summary.py).  A kernel added later without a case fails the gate.

Every SpMV case runs twice: once with finite inputs, once with the same rows where x and A carry +-Inf, NaN (with
and without payload), subnormals and signed zeros placed where the work is split (merge-tile boundaries, window
boundaries, rows spanning tiles, the unstaged tail of the non-zeros, the most referenced column), and with a NaN in
x at column 0 and at the last column that no row references -- a kernel that gathers x[0] for a padding slot turns
rows into NaN.  Finite magnitudes stay <= 1e30, so no fp32 overflow depends on the summation order.

Rules: "exact" -- the kernels that keep spmv_cpu_csr's front-to-back order (SCALAR family, one-lane VECTOR, every
ELL form, the host-buffer forms, plan mode 5) are bit-identical to the oracle, NaN counted as one value;
"order_free" -- the reordering kernels are NaN and +-Inf exactly where the oracle is, and every other row within
1e-5 * sum_j |a_ij x_j| of the f64 oracle; "hub" -- order_free and bit-identical to plain MERGE_PATH."""
import ctypes as C
import functools
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-spmv_b200", "lib", "libspmv_b200.so")


def _sass_summary():
    spec = importlib.util.spec_from_file_location("sass_summary", os.path.join(ROOT, "scripts", "sass_summary.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------ matrices ----
# (rows, cols, row_ptrs, col_indices, values) in numpy; deterministic per seed.

def _csr_from_lens(lens, cols, rng, col_of=None):
    lens = np.asarray(lens, np.int64)
    rp = np.zeros(len(lens) + 1, np.int64)
    rp[1:] = np.cumsum(lens)
    nnz = int(rp[-1])
    row = np.repeat(np.arange(len(lens)), lens)
    ci = rng.integers(0, cols, nnz) if col_of is None else col_of(row, rp)
    order = np.lexsort((ci, row))
    va = rng.uniform(-1, 1, nnz).astype(np.float32)
    return len(lens), cols, rp.astype(np.int32), ci[order].astype(np.int32), va


def m_random(rows, cols, avg, seed, long_rows=0, long_len=6000):
    """Row lengths uniform in [0, 2 avg]; `long_rows` rows of `long_len` non-zeros spread over the matrix."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 2 * avg + 1, rows)
    for i in range(long_rows):
        lens[(i * 7919 + rows // 3) % rows] = long_len
    return _csr_from_lens(lens, cols, rng)


def m_uniform(rows, k, cols, seed):
    """Exactly k distinct columns in every row."""
    rng = np.random.default_rng(seed)

    def col_of(row, rp):
        base = rng.integers(0, cols - k, len(rp) - 1)
        return base[row] + (np.arange(len(row)) - rp[row])
    return _csr_from_lens(np.full(rows, k), cols, rng, col_of)


def m_stencil(grid, points, seed):
    """5- or 9-point stencil on a grid x grid mesh (boundary rows are shorter)."""
    offs = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)] + ([(-1, -1), (-1, 1), (1, -1), (1, 1)] if points == 9 else [])
    n = grid * grid
    i = np.arange(n)
    gy, gx = i // grid, i % grid
    rows_l, cols_l = [], []
    for dy, dx in offs:
        ok = (gy + dy >= 0) & (gy + dy < grid) & (gx + dx >= 0) & (gx + dx < grid)
        rows_l.append(i[ok])
        cols_l.append((gy[ok] + dy) * grid + gx[ok] + dx)
    r, c = np.concatenate(rows_l), np.concatenate(cols_l)
    order = np.lexsort((c, r))
    rp = np.zeros(n + 1, np.int32)
    rp[1:] = np.cumsum(np.bincount(r, minlength=n))
    va = np.random.default_rng(seed).uniform(-1, 1, len(c)).astype(np.float32)
    return n, n, rp, c[order].astype(np.int32), va


def m_banded(rows, w, seed):
    """Row i reads columns i - w/2 .. i + w/2 - 1 inside the matrix: w per row, fewer (ELL padding) at the edges."""
    rng = np.random.default_rng(seed)
    lo = np.clip(np.arange(rows) - w // 2, 0, None)
    hi = np.clip(np.arange(rows) - w // 2 + w, None, rows)
    lens = hi - lo

    def col_of(row, rp):
        return lo[row] + (np.arange(len(row)) - rp[row])
    return _csr_from_lens(lens, rows, rng, col_of)


def m_max_width(rows, w, seed):
    """Random rows of 0 .. w non-zeros, at least one row of exactly w."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, w + 1, rows)
    lens[rows // 2] = w
    return _csr_from_lens(lens, rows, rng)


def m_rmat(scale, ef, seed):
    import gpu_spmv_b200.gen as gen
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, ef, seed, "cpu")
    return n, n, rp.numpy(), ci.numpy(), va.numpy()


# ---------------------------------------------------------------------------------------------- IEEE inputs ----
NAN_PAYLOAD = np.array([0x7FC0BEEF], np.uint32).view(np.float32)[0]
SUB_X, SUB_A = np.float32(1e-40), np.float32(3e-39)


def ieee_inputs(m, x):
    """The same rows with specials in x and A where the work is split.  Columns move up by one and two
    columns are added, 0 and cols + 1, that no row references; x holds NaN there."""
    rows, cols, rp, ci, va = m
    nnz = len(ci)
    ci2, va2 = ci + 1, va.copy()
    x2 = np.empty(cols + 2, np.float32)
    x2[1:-1] = x
    x2[0] = x2[-1] = np.float32(np.nan)
    pos = set(range(max(nnz - 3, 0), nnz))                      # the unstaged tail
    for t in (256 * 7, 256 * 8):                                # first / last non-zero of merge tiles
        for k in range(t, nnz + 1, t):
            pos.update((k - 1, k, k + 1))
    for w in (256, 512):                                        # first / last non-zero of windows
        for r in range(w, rows, w):
            pos.update((int(rp[r]) - 1, int(rp[r])))
    lens = np.diff(rp)
    for r in np.flatnonzero(lens > 256 * 7)[:8]:                # rows that span tiles
        pos.update((int(rp[r]), int(rp[r] + lens[r] // 2), int(rp[r + 1]) - 1))
    pos = sorted(p for p in pos if 0 <= p < nnz)
    special_cols = set()
    # a special x entry reaches every row that reads its column: keep those rows near a tenth of the matrix,
    # with the special columns spread over all the positions
    max_x = max(4, int(0.1 * rows * cols / max(nnz, 1)))
    x_every = -(-len(pos) * 7 // 13 // max_x) or 1
    x_calls = [0]

    def set_x(p, v):
        c = int(ci2[p])
        x_calls[0] += 1
        if c not in special_cols and x_calls[0] % x_every == 0:
            special_cols.add(c)
            x2[c] = v
    for i, p in enumerate(pos):
        k = i % 13
        if k == 0:
            va2[p] = SUB_A
        elif k == 1:  # a stored +0.0 on an Inf column: 0 * Inf = NaN
            va2[p] = 0.0
            set_x(p, np.inf)
        elif k == 2:
            va2[p] = np.float32(1e30) if i % 2 else np.float32(-1e30)
        elif k == 3:
            set_x(p, SUB_X)
        elif k == 4:
            va2[p] = np.float32(-0.0)
        elif k == 5:  # a stored -0.0 on a -Inf column
            va2[p] = np.float32(-0.0)
            set_x(p, -np.inf)
        elif k == 6:
            va2[p] = -SUB_A
        elif k == 7:
            set_x(p, np.nan)
        elif k == 8:  # a subnormal product of two normal numbers
            va2[p] = np.float32(1e-20)
            set_x(p, np.float32(3e-21))
        elif k == 9:
            set_x(p, np.float32(-0.0))
        elif k == 10:
            set_x(p, NAN_PAYLOAD)
        elif k == 11:
            set_x(p, np.inf)
        else:
            set_x(p, -np.inf)
    if nnz:  # the most referenced column (the hub table's first entry)
        hub = int(np.argmax(np.bincount(ci2, minlength=cols + 2)))
        if hub not in special_cols:
            x2[hub] = -SUB_X
    return (rows, cols + 2, rp, ci2.astype(np.int32), va2), x2


# ----------------------------------------------------------------------------------------------- the cases ----
class Case:
    def __init__(self, name, env, build, entry, expect, rule="exact", **opts):
        self.name, self.env, self.build, self.entry = name, dict(env), build, entry
        self.expect = tuple(expect)  # every entry must run; "a|b": one of them
        self.rule, self.opts = rule, opts

    @property
    def group(self):
        return json.dumps(self.env, sort_keys=True)


def _pipe(lpr, u, robust):
    return f"csr_pipe_kernel<{lpr}, {u}, {'true' if robust else 'false'}>"


def _cases():
    c = []
    V = "SPMV_B200_"
    # -- row-owner rings: LPR from SCALAR (1) or SPMV_B200_VECTOR_LANES, U from the load per lane
    #    (<= 4 / <= 6 / more), ROBUST by structure: a 6000-entry row is longer than half a stage and its
    #    window overflows the stage (pipe_overflow_window)
    for lpr in (1, 2, 4, 8, 16):
        env = {} if lpr == 1 else {V + "VECTOR_LANES": str(lpr)}
        entry = "SCALAR" if lpr == 1 else "VECTOR"
        rule = "exact" if lpr == 1 else "order_free"
        for u, per_lane in ((4, 3), (6, 5), (8, 7)):
            avg = per_lane * lpr
            rows = int(np.clip(200000 // avg, 1500, 20000))
            for robust in (False, True):
                c.append(Case(f"pipe_lpr{lpr}_u{u}_{'robust' if robust else 'fast'}", env,
                              functools.partial(m_random, rows, rows, avg, 100 * lpr + u, 3 if robust else 0),
                              entry, [_pipe(lpr, u, robust)], rule))
        if lpr > 1:  # pointers that are only 4-byte aligned take the register-staged kernel
            c.append(Case(f"stream_lpr{lpr}_unaligned", env, functools.partial(m_random, 3000, 3000, 3 * lpr, 7 + lpr),
                          "VECTOR", [f"csr_stream_kernel<{lpr}>"], "order_free", unaligned=True))
    c.append(Case("stream_lpr1_unaligned", {}, functools.partial(m_random, 3000, 3000, 5, 8), "SCALAR",
                  ["csr_stream_kernel<1>"], unaligned=True))
    for lanes, avg in ((1, 5), (8, 25), (16, 40)):
        c.append(Case(f"stream_lpr{lanes}_no_pipe", {V + "CSR_NO_PIPE": "1"},
                      functools.partial(m_random, 4000, 4000, avg, 30 + lanes), "SCALAR" if lanes == 1 else "VECTOR",
                      [f"csr_stream_kernel<{lanes}>"], "exact" if lanes == 1 else "order_free"))
    for stages in ("3", "16"):  # 16 stages may not fit the 200 KiB guard: then the register-staged kernel
        env = {V + "CSR_STAGES": stages}
        alt = "" if stages == "3" else "|csr_stream_kernel<1>"
        c.append(Case(f"pipe_stages{stages}_lpr1", env, functools.partial(m_random, 20000, 20000, 5, 41), "SCALAR",
                      [_pipe(1, 6, False) + alt]))
        alt = "" if stages == "3" else "|csr_stream_kernel<8>"
        c.append(Case(f"pipe_stages{stages}_lpr8", env, functools.partial(m_random, 6000, 6000, 25, 42), "VECTOR",
                      [_pipe(8, 4, False) + alt], "order_free"))
        c.append(Case(f"pipe_stages{stages}_robust", env, functools.partial(m_random, 20000, 20000, 3, 43, 2), "SCALAR",
                      [_pipe(1, 4, True) + ("" if stages == "3" else "|csr_stream_kernel<1>")]))
    c.append(Case("pipe_rpg8_lpr1", {V + "CSR_RPG": "8"}, functools.partial(m_random, 20000, 20000, 3, 44), "SCALAR",
                  [_pipe(1, 4, False)]))
    c.append(Case("pipe_rpg8_lpr8", {V + "CSR_RPG": "8"}, functools.partial(m_random, 6000, 6000, 25, 45), "VECTOR",
                  [_pipe(8, 4, False)], "order_free"))
    c.append(Case("warp_row", {}, functools.partial(m_random, 1500, 8000, 70, 46), "VECTOR", ["csr_warp_row_kernel"],
                  "order_free"))
    # -- short-row ring: uniform rows, a partial last window, nnz % 4 != 0
    c.append(Case("short_2_per_row", {}, functools.partial(m_uniform, 2637, 2, 5000, 47), "SCALAR",
                  ["csr_short_kernel<4, 2, 1536, 2>"]))
    c.append(Case("short_laplacian", {}, functools.partial(m_stencil, 101, 5, 48), "SCALAR",
                  ["csr_short_kernel<6, 1, 1536, 2>"]))
    c.append(Case("short_9_point", {}, functools.partial(m_stencil, 103, 9, 49), "SCALAR",
                  ["csr_short_kernel<8, 1, 3072, 2>"]))
    c.append(Case("short_9_point_vector", {}, functools.partial(m_stencil, 103, 9, 50), "VECTOR",
                  ["csr_short_kernel<8, 1, 3072, 2>"]))
    c.append(Case("short_forced_dense_window", {V + "CSR_SHORT": "1"},
                  functools.partial(m_random, 20000, 20000, 1, 51, 2, 3000), "SCALAR", ["csr_short_kernel<4, 2, 1536, 2>"]))
    # -- ELL: the kernel by row count and width, SPMV_B200_ELL_VARIANT 1-5, ring depth
    c.append(Case("ell_pipe1_w8", {}, functools.partial(m_banded, 4000, 8, 52), "ELL", ["ell_tma_pipe_kernel<1>"]))
    c.append(Case("ell_pipe1_w1", {}, functools.partial(m_uniform, 4000, 1, 4000, 53), "ELL", ["ell_tma_pipe_kernel<1>"]))
    c.append(Case("ell_tma2_w9", {}, functools.partial(m_max_width, 4000, 9, 54), "ELL", ["ell_tma_kernel<2>"]))
    c.append(Case("ell_slice1_odd_rows", {}, functools.partial(m_max_width, 4001, 8, 55), "ELL", ["ell_slice_kernel<1>"]))
    c.append(Case("ell_slice2_even_rows", {}, functools.partial(m_max_width, 4002, 9, 56), "ELL", ["ell_slice_kernel<2>"]))
    for variant, kernel in (("1", "ell_slice_kernel<4>"), ("2", "ell_tma_kernel<4>"), ("3", "ell_tma_kernel<2>"),
                            ("4", "ell_tma_pipe_kernel<4>"), ("5", "ell_tma_pipe_kernel<2>")):
        c.append(Case(f"ell_variant{variant}_w8", {V + "ELL_VARIANT": variant}, functools.partial(m_max_width, 4000, 8, 57),
                      "ELL", [kernel]))
    c.append(Case("ell_variant4_w1", {V + "ELL_VARIANT": "4"}, functools.partial(m_uniform, 4000, 1, 4000, 58), "ELL",
                  ["ell_tma_pipe_kernel<4>"]))
    c.append(Case("ell_stages3_w8", {V + "ELL_STAGES": "3"}, functools.partial(m_banded, 20000, 8, 59), "ELL",
                  ["ell_tma_pipe_kernel<1>"]))
    # 16 stages of W = 8 do not fit one CTA's shared memory: the ring is cut to what fits
    env16 = {V + "ELL_STAGES": "16", V + "HOST_GATED": "0"}
    c.append(Case("ell_stages16_w8", env16, functools.partial(m_banded, 20000, 8, 60), "ELL", ["ell_tma_pipe_kernel<1>"]))
    c.append(Case("ell_host_chunked_stages16_w8", env16, functools.partial(m_banded, 65536, 8, 61), "HOST",
                  ["ell_tma_pipe_kernel<1>", "ell_chunk_col_range_kernel"], chunks=8, gated=False))
    c.append(Case("ell_variant4_stages16_w8", {V + "ELL_VARIANT": "4", V + "ELL_STAGES": "16"},
                  functools.partial(m_banded, 20000, 8, 62), "ELL", ["ell_tma_pipe_kernel<4>"]))
    c.append(Case("ell_host_gated", {}, functools.partial(m_stencil, 256, 5, 63), "HOST", ["ell_tma_gated_kernel"],
                  chunks=0, gated=True))
    # -- merge-path: 8 items per thread for 4 <= avg < 10, else 7; SPMV_B200_MERGE_IPT / _TMA force
    c.append(Case("merge_ipt8", {}, functools.partial(m_random, 30000, 30000, 5, 64), "MERGE",
                  ["merge_tile_kernel<PlainRow, 8>", "merge_partition_kernel", "merge_fixup_kernel<PlainRow>"], "order_free"))
    c.append(Case("merge_ipt7", {}, functools.partial(m_random, 20000, 20000, 12, 65), "MERGE",
                  ["merge_tile_kernel<PlainRow, 7>"], "order_free"))
    c.append(Case("merge_rows_span_tiles", {}, functools.partial(m_random, 20000, 20000, 2, 66, 3, 20000), "MERGE",
                  ["merge_tile_kernel<PlainRow, 8>"], "order_free"))
    c.append(Case("merge_forced_ipt7", {V + "MERGE_IPT": "7"}, functools.partial(m_random, 30000, 30000, 5, 67), "MERGE",
                  ["merge_tile_kernel<PlainRow, 7>"], "order_free"))
    c.append(Case("merge_forced_ipt8", {V + "MERGE_IPT": "8"}, functools.partial(m_random, 20000, 20000, 12, 68), "MERGE",
                  ["merge_tile_kernel<PlainRow, 8>"], "order_free"))
    for avg, ipt in ((5, 8), (12, 7)):
        c.append(Case(f"merge_tma_ipt{ipt}", {V + "MERGE_TMA": "1"}, functools.partial(m_random, 20000, 20000, avg, 69 + avg),
                      "MERGE", [f"merge_tile_kernel<PlainRow, {ipt}>"], "order_free"))
        # hub-column kernel: a 64-entry table, and all of x in shared memory (cap 0 = device maximum)
        c.append(Case(f"hub_table_ipt{ipt}", {}, functools.partial(m_random, 20000, 20000, avg, 71 + avg, 2, 5000), "PLAN",
                      [f"merge_hot_kernel<PlainRow, false, {ipt}>"], "hub", cap=64, modes=(1,)))
        c.append(Case(f"hub_all_x_ipt{ipt}", {}, functools.partial(m_random, 20000, 20000, avg, 73 + avg), "PLAN",
                      [f"merge_hot_kernel<PlainRow, true, {ipt}>"], "hub", cap=0, modes=(2,)))
    seg = {V + "PLAN": "seg", V + "HOT": "1", V + "PR_SMALL": "0"}
    c.append(Case("seg_table", seg, functools.partial(m_random, 30000, 30000, 6, 75), "PLAN",
                  ["seg_spmv_kernel", "seg_fixup_kernel"], "order_free", cap=64, modes=(3, 4)))
    c.append(Case("seg_rows_span_tiles", seg, functools.partial(m_random, 20000, 20000, 5, 76, 3, 20000), "PLAN",
                  ["seg_spmv_kernel", "seg_fixup_kernel"], "order_free", cap=64, modes=(3, 4)))
    c.append(Case("plan_ell_snapshot", {}, functools.partial(m_stencil, 100, 5, 77), "PLAN",
                  ["ell_from_csr_kernel", "ell_tma_pipe_kernel<1>"], snapshot=True, modes=(5,)))
    # -- everything else: one cheap call each, finite inputs, checked as the existing tests do
    c.append(Case("zero_rows", {}, None, "ZERO", ["zero_rows_kernel"], "misc"))
    c.append(Case("pagerank_small", {}, functools.partial(m_rmat, 10, 8, 3), "PAGERANK", ["pagerank_small_kernel"], "misc"))
    c.append(Case("pagerank_api", {}, functools.partial(m_rmat, 11, 8, 4), "PAGERANK_API", [], "misc"))
    c.append(Case("pagerank_tile", {V + "HOT": "0", V + "PR_SMALL": "0"}, functools.partial(m_rmat, 12, 8, 5), "PAGERANK",
                  ["merge_tile_kernel<PageRankRowT<false>, 7>", "merge_fixup_kernel<PageRankRowT<false>>"], "misc"))
    c.append(Case("pagerank_seg", seg, functools.partial(m_rmat, 12, 8, 6), "PAGERANK", ["seg_pagerank_epilogue_kernel"],
                  "misc"))
    hub = {V + "PLAN": "hub", V + "HOT": "1", V + "PR_SMALL": "0"}
    c.append(Case("pagerank_hub_all_x", hub, functools.partial(m_rmat, 12, 8, 7), "PAGERANK",
                  ["merge_hot_kernel<PageRankRowT<true>, true, 7>"], "misc"))
    c.append(Case("pagerank_hub_table", hub, functools.partial(m_rmat, 17, 4, 8), "PAGERANK",
                  ["merge_hot_kernel<PageRankRowT<true>, false, 7>"], "misc"))
    c.append(Case("top_k_device", {}, None, "TOPK", ["topk_hist_kernel", "topk_tie_write_kernel"], "misc"))
    c.append(Case("coo_assembly_and_normalisation", {}, None, "COO", ["coo_keys_kernel", "coo_row_ptrs_kernel",
                                                                      "divide_by_colsum_kernel"], "misc"))
    c.append(Case("h2d_order_probe", {}, None, "PROBE", ["probe_arrival_kernel"], "misc"))
    return c


CASES = _cases()
GROUPS = sorted({c.group for c in CASES}, key=lambda g: (g != "{}", g))

# Shipped kernels no case here launches, with the reason.
NOT_RUN_HERE = {
    "cub::CUB_200802_SM_1000::EmptyKernel<void>": "never launched: CUB's placeholder for querying PTX versions",
    "merge_tile_kernel<PageRankRowT<false>, 8>":
        "unreachable: PageRank merge plans are always cut at 7 items per thread (pagerank.cu, merge_plan_carve)",
    "pr_count_kernel": "multi-rank PageRank exchange: tests/test_gpu_multi_one_device.py",
    "pr_gate_kernel": "multi-rank PageRank exchange: tests/test_gpu_multi_one_device.py",
    "pr_publish_kernel": "multi-rank PageRank exchange: tests/test_gpu_multi_one_device.py",
    "pr_sum_peers_kernel": "multi-rank PageRank exchange: tests/test_gpu_multi_one_device.py",
}


# ------------------------------------------------------------------------------------------------- checks ----
def check_result(rule, y, ref32, ref64, scale, what):
    from gpu_helpers import assert_same_bits_nan_as_class
    if rule == "exact":
        assert_same_bits_nan_as_class(y, ref32, what)
        return
    nan_r, nan_y = np.isnan(ref32), np.isnan(y)
    assert np.array_equal(nan_y, nan_r), f"{what}: NaN in {int((nan_y & ~nan_r).sum())} rows the oracle has not, " \
        f"missing in {int((nan_r & ~nan_y).sum())} rows (first {np.flatnonzero(nan_y != nan_r)[:5].tolist()})"
    inf_r = np.isinf(ref32)
    bad = np.flatnonzero((np.isinf(y) != inf_r) | (inf_r & (y != ref32)))
    assert bad.size == 0, f"{what}: +-Inf differs from the oracle in {bad.size} rows, first {bad[0]}: {y[bad[0]]} vs {ref32[bad[0]]}"
    fin = ~nan_r & ~inf_r
    err = np.abs(y[fin].astype(np.float64) - ref64[fin])
    out = err > 1e-5 * scale[fin] + 1e-30
    assert not out.any(), f"{what}: {int(out.sum())} rows out of tolerance, worst {err[out].max()}"


# ------------------------------------------------------------------------------------------ child process ----
class _Runner:
    def __init__(self):
        import torch
        sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
        from _load_pkg import load_pkg
        from oracle_binding import Oracle
        self.torch, self.sp, self.orc = torch, load_pkg(), Oracle()
        torch.cuda.set_device(0)
        self.dev = torch.device("cuda:0")

    def t(self, a, unaligned=False):
        a = self.torch.as_tensor(np.ascontiguousarray(a))
        if not unaligned:
            return a.to(self.dev)
        return self.torch.cat([a.new_zeros(1), a]).to(self.dev)[1:]

    def device_csr(self, m, unaligned=False):
        rows, cols, rp, ci, va = m
        return self.sp.DeviceCSR(rows, cols, self.t(rp, unaligned), self.t(ci, unaligned), self.t(va, unaligned))

    def host_ell(self, m):
        sp = self.sp
        rows, cols, rp, ci, va = m
        A = sp.csr_from_arrays(rows, cols, rp, ci, va)
        E = sp.ell_create(0, 0, 0)
        assert sp.ell_from_csr(E, A) == 0 and sp.ell_to_gpu(E) == 0
        sp.csr_destroy(A)
        ec, ev = sp.ell_arrays(E)
        return E, E.contents.max_nnz_per_row, ec.copy(), ev.copy()

    def spmv(self, case, m, x):
        """y of the case's entry point, and the sequential-order oracle for it."""
        sp, torch = self.sp, self.torch
        rows, cols, rp, ci, va = m
        d_x = self.t(x.astype(np.float32))
        d_y = torch.full((rows,), float("nan"), dtype=torch.float32, device=self.dev)
        ref32 = self.orc.spmv_csr(rows, rp, ci, va, x)
        e = case.entry
        if e in ("SCALAR", "VECTOR", "MERGE"):
            A = self.device_csr(m, case.opts.get("unaligned", False))
            if case.opts.get("unaligned"):
                d_x, d_y = self.t(x.astype(np.float32), True), torch.full((rows + 1,), float("nan"), device=self.dev)[1:]
            k = {"SCALAR": sp.SCALAR_CSR, "VECTOR": sp.VECTOR_CSR, "MERGE": sp.MERGE_PATH}[e]
            res = sp.spmv_csr(A.ptr, d_x, d_y, sp.make_config(k), cols)
            assert res.error_code == 0, f"spmv_csr returned {res.error_code}"
        elif e == "ELL":
            E, w, ec, ev = self.host_ell(m)
            res = sp.spmv_ell(E, d_x, d_y, None, cols)
            sp.ell_destroy(E)
            assert res.error_code == 0, f"spmv_ell returned {res.error_code}"
            ref32 = self.orc.spmv_ell(rows, w, ec, ev, x)
        elif e == "HOST":
            E, w, ec, ev = self.host_ell(m)
            plan = C.c_void_p()
            assert sp.lib.spmv_b200_ell_host_plan_create(E, case.opts["chunks"], C.byref(plan)) == 0
            gated = C.c_int()
            assert sp.lib.spmv_b200_ell_host_plan_gated(plan, C.byref(gated), None) == 0
            assert gated.value == int(case.opts["gated"]), f"gated form {gated.value}"
            xh = torch.as_tensor(x.astype(np.float32)).pin_memory()
            yh = torch.full((rows,), float("nan")).pin_memory()
            rc = sp.lib.spmv_b200_spmv_ell_host(plan, xh.data_ptr(), yh.data_ptr())
            sp.lib.spmv_b200_ell_host_plan_destroy(plan)
            sp.ell_destroy(E)
            assert rc == 0, f"spmv_ell_host returned {rc}"
            d_y = yh
            ref32 = self.orc.spmv_ell(rows, w, ec, ev, x)
        elif e == "PLAN":
            A = self.device_csr(m)
            plan = sp.CsrPlan(A.ptr, case.opts.get("cap", 0), force=not case.opts.get("snapshot"),
                              snapshot_values=bool(case.opts.get("snapshot")))
            mode = plan.info()[2]
            assert mode in case.opts["modes"], f"plan mode {mode}"
            assert plan.spmv(d_x, d_y) == 0
            torch.cuda.synchronize()
            plan.close()
            if case.rule == "hub":  # the table only changes where x[col] is read from
                y_plain = torch.full((rows,), float("nan"), dtype=torch.float32, device=self.dev)
                assert sp.spmv_csr(A.ptr, d_x, y_plain, sp.make_config(sp.MERGE_PATH), cols).error_code == 0
                self.y_plain = y_plain.cpu().numpy()
        else:
            raise ValueError(e)
        torch.cuda.synchronize()
        return d_y.cpu().numpy()[:rows], ref32

    def run_spmv_case(self, case):
        from gpu_helpers import assert_same_bits_nan_as_class
        m = case.build()
        x = np.random.default_rng(len(case.name)).uniform(-1, 1, m[1]).astype(np.float32)
        for label, (mm, xx) in (("finite", (m, x)), ("ieee", ieee_inputs(m, x))):
            y, ref32 = self.spmv(case, mm, xx)
            rows, cols, rp, ci, va = mm
            ref64, scale = self.orc.spmv_csr_f64(rows, rp, ci, va, xx)
            check_result("exact" if case.rule == "exact" else "order_free", y, ref32, ref64, scale, f"{case.name} {label}")
            if case.rule == "hub":
                assert_same_bits_nan_as_class(y, self.y_plain, f"{case.name} {label}: hub plan against plain MERGE_PATH")

    def run_misc_case(self, case):
        sp, torch, orc, dev = self.sp, self.torch, self.orc, self.dev
        e = case.entry
        if e == "ZERO":
            Z = sp.DeviceCSR(37, 5, torch.zeros(38, dtype=torch.int32, device=dev), torch.zeros(4, dtype=torch.int32, device=dev),
                             torch.zeros(4, device=dev), nnz=0)
            d_y = torch.full((37,), float("nan"), device=dev)
            assert sp.spmv_csr(Z.ptr, torch.ones(5, device=dev), d_y, sp.make_config(sp.SCALAR_CSR), 5).error_code == 0
            assert not d_y.cpu().numpy().any()
        elif e == "PAGERANK":
            m = case.build()
            n, _, rp, ci, va = m
            G = self.device_csr(m)
            d_ranks = torch.empty(n, dtype=torch.float32, device=dev)
            rc, iters, res, conv, l1 = sp.pagerank_device(G.ptr, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100))
            assert rc == 0 and iters > 0, (rc, iters)
            o_ranks = orc.pagerank_f64(n, n, rp, ci, va, 0.85, 1e-6, 100, fixed_it=iters)[0]
            l1_err = np.abs(d_ranks.cpu().numpy().astype(np.float64) - o_ranks).sum()
            assert l1_err <= 1e-6, f"L1 {l1_err} after {iters} iterations"
        elif e == "PAGERANK_API":
            n, _, rp, ci, va = case.build()
            G = sp.csr_from_arrays(n, n, rp, ci, va)
            assert sp.csr_to_gpu(G) == 0
            result, ranks = sp.pagerank(G, sp.make_pagerank_config(0.85, 1e-6, 100))
            l_ranks, l_it = orc.pagerank_f32(n, n, rp, ci, va, 0.85, 1e-6, 100)[:2]
            assert abs(result.iterations - l_it) <= 1 and np.abs(ranks.astype(np.float64) - l_ranks).sum() <= 2e-6
            sp.pagerank_free(result)
            sp.csr_destroy(G)
        elif e == "TOPK":  # few distinct values: the threshold falls inside a long run of equal ranks
            n, k = 300000, 1000
            v = (np.random.default_rng(5).integers(0, 12, n) / 16.0).astype(np.float32)
            ids, vals = sp.pagerank_top_k_device(torch.as_tensor(v).to(dev), k)
            assert np.array_equal(vals, sp.pagerank_top_k(v, k)[1])
            expect = np.lexsort((np.arange(n), -v.astype(np.float64)))[:k]  # rank descending, id ascending
            assert np.array_equal(ids, expect.astype(np.int32))
        elif e == "COO":
            import gpu_spmv_b200.gen as gen
            # a few entries (one-tile sort), duplicates keep their input order
            rng = np.random.default_rng(3)
            r, c = rng.integers(0, 50, 300).astype(np.int32), rng.integers(0, 40, 300).astype(np.int32)
            r[1::7], c[1::7] = r[0], c[0]
            v = rng.uniform(-1, 1, 300).astype(np.float32)
            A = sp.csr_create(0, 0, 0)
            assert sp.csr_from_coo_device(A, 50, 40, self.t(r), self.t(c), self.t(v)) == 0 and sp.csr_from_gpu(A) == 0
            order = np.lexsort((c, r))
            g_rp, g_ci, g_va = sp.csr_arrays(A)
            assert np.array_equal(g_rp[1:], np.cumsum(np.bincount(r, minlength=50))) and np.array_equal(g_ci, c[order])
            assert np.array_equal(g_va.view(np.uint32), v[order].view(np.uint32))
            sp.csr_destroy(A)
            n, rp, ci, va = gen.rmat_pagerank_csr(11, 8, 9, "cpu")
            src, dst = gen.rmat_edges(11, 8, 9, dev)
            A = sp.csr_create(0, 0, 0)
            assert sp.csr_from_coo_device(A, n, n, dst.to(torch.int32), src.to(torch.int32),
                                          torch.ones(src.numel(), device=dev)) == 0
            assert sp.csr_normalize_columns_device(A) == 0 and sp.csr_from_gpu(A) == 0
            g_rp, g_ci, g_va = sp.csr_arrays(A)
            assert np.array_equal(g_rp, rp.numpy()) and np.array_equal(g_ci, ci.numpy())
            assert np.array_equal(g_va.view(np.uint32), va.numpy().view(np.uint32))
            sp.csr_destroy(A)
        elif e == "PROBE":
            xh = torch.rand(1 << 20).pin_memory()
            out = (C.c_longlong * 9)()
            assert sp.lib.spmv_b200_probe_h2d_order(xh.data_ptr(), 1 << 20, 8, out, 1, 0) == 0
            assert min(list(out)[:8]) == 0
        else:
            raise ValueError(e)

    def kernels_of(self, fn):
        from torch.autograd import DeviceType
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            self.torch.cuda.synchronize()
        names = sorted({ev.name for ev in prof.events() if ev.device_type == DeviceType.CUDA})
        return [n for n in _sass_summary().demangle(names) if not n.startswith(("Memcpy", "Memset"))] if names else []


def child_main(group):
    import traceback
    r = _Runner()
    for case in CASES:
        if case.group != group:
            continue
        ok, msg = True, ""

        def run():
            if case.rule == "misc":
                r.run_misc_case(case)
            else:
                r.run_spmv_case(case)
        try:
            kernels = r.kernels_of(run)
        except Exception as exc:  # noqa: BLE001 -- reported to the parent, case by case
            ok, msg, kernels = False, f"{type(exc).__name__}: {exc}\n{traceback.format_exc()[-1500:]}", []
        print("CASE " + json.dumps({"case": case.name, "ok": ok, "msg": msg, "kernels": kernels}), flush=True)


@functools.lru_cache(maxsize=None)
def run_group(group):
    env = {k: v for k, v in os.environ.items() if not k.startswith("SPMV_B200_")}
    env.update(json.loads(group))
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", group], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    out = {}
    for line in p.stdout.splitlines():
        if line.startswith("CASE "):
            rec = json.loads(line[5:])
            out[rec["case"]] = rec
    return p.returncode, p.stdout, out


# ---------------------------------------------------------------------------------------------------- tests ----
def _needs_lib():
    if not os.path.exists(LIB):
        pytest.skip("libspmv_b200.so is not built")


def test_expected_kernel_names_are_shipped():
    """Every kernel a case expects, and every NOT_RUN_HERE entry, exists in the built library (catches typos and
    renames; cuobjdump only, no GPU)."""
    _needs_lib()
    shipped = _sass_summary().shipped_kernels(LIB)
    missing = sorted({alt for c in CASES for e in c.expect for alt in e.split("|") if alt not in shipped} |
                     {k for k in NOT_RUN_HERE if k not in shipped})
    assert not missing, f"not in libspmv_b200.so: {missing}"
    assert len({c.name for c in CASES}) == len(CASES)


def _group_id(group):
    return ",".join(f"{k[len('SPMV_B200_'):]}={v}" for k, v in json.loads(group).items()) or "defaults"


@pytest.mark.gpu
@pytest.mark.parametrize("group", GROUPS, ids=_group_id)
def test_kernel_cases(cuda, group):
    rc, stdout, recs = run_group(group)
    cases = [c for c in CASES if c.group == group]
    assert rc == 0 and len(recs) == len(cases), stdout[-4000:]
    failed = [f"{r['case']}: {r['msg']}" for r in recs.values() if not r["ok"]]
    assert not failed, "\n".join(failed)
    if not any(r["kernels"] for r in recs.values()):
        return  # the profiler records no CUDA kernels here: the coverage gate reports it
    wrong = []
    for c in cases:
        seen = set(recs[c.name]["kernels"])
        for e in c.expect:
            if not seen & set(e.split("|")):
                wrong.append(f"{c.name}: expected {e}, ran {sorted(seen)}")
        print(f"{c.name}: {sorted(seen)}")
    assert not wrong, "\n".join(wrong)


@pytest.mark.gpu
def test_coverage_gate(cuda):
    """observed kernels + NOT_RUN_HERE == the kernels libspmv_b200.so ships."""
    shipped = _sass_summary().shipped_kernels(LIB)
    observed = set()
    for g in GROUPS:
        observed |= {k for r in run_group(g)[2].values() for k in r["kernels"]}
    if not observed:
        pytest.skip("torch.profiler recorded no CUDA kernels on this machine: kernel coverage not measured")
    seen = observed & shipped
    print(f"\nshipped {len(shipped)}, observed {len(seen)}, NOT_RUN_HERE {len(NOT_RUN_HERE)}")
    for k in sorted(shipped):
        print(f"  {'observed' if k in seen else 'NOT_RUN_HERE: ' + NOT_RUN_HERE.get(k, '-- MISSING --')} | {k}")
    missing = sorted(shipped - seen - set(NOT_RUN_HERE))
    stale = sorted(k for k in NOT_RUN_HERE if k not in shipped)
    assert not missing and not stale, f"shipped but never run: {missing}; listed but not shipped: {stale}"


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    child_main(sys.argv[2])
