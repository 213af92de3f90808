"""CSR plans: the planned kernels that keep the x entries of the most referenced columns in shared
memory -- the segmented-stream kernel (csr_seg_kernels.cu, default) and the hub-column merge-path
kernel (csr_hot_kernels.cu, SPMV_B200_PLAN=hub).

Every result must be within the north_star tolerance of the oracle (|y - y_ref| <= 1e-5 *
sum_j |a_ij x_j| per row against the f64-accumulating restatement of spmv_cpu_csr, reference
src/spmv_cpu.cpp:6-16), deterministic (two products give the same bits), and -- for the
hub-column merge-path kernel, which only changes WHERE x[col] is read from -- BIT-IDENTICAL to
spmv_csr(MERGE_PATH) without a plan."""
import os

import numpy as np
import pytest
import torch

from gpu_helpers import assert_within_tolerance, bits

pytestmark = pytest.mark.gpu
MERGE = 2
SEG = os.environ.get("SPMV_B200_PLAN", "").startswith("s")  # the segmented-stream kernel is forced
HUB = not SEG  # scale-free inputs (and force=True) get the hub-column merge-path kernel by default


def gen_mod():
    import gpu_spmv_b200.gen as gen
    return gen


def plain_merge(sp, A, d_x, rows, cols):
    d_y = torch.full((max(rows, 1),), float("nan"), dtype=torch.float32, device=d_x.device)
    res = sp.spmv_csr(A.ptr, d_x, d_y, sp.make_config(MERGE), cols)
    assert res.error_code == 0
    return d_y[:rows].cpu().numpy()


def check_plan(sp, orc, dev, rows, cols, rp, ci, va, x, caps, what, expect_mode=None):
    rp, ci, va, x = (np.ascontiguousarray(rp, np.int32), np.ascontiguousarray(ci, np.int32),
                     np.ascontiguousarray(va, np.float32), np.ascontiguousarray(x, np.float32))
    y64, scale = orc.spmv_csr_f64(rows, rp, ci, va, x)
    t = lambda a: torch.as_tensor(a).to(dev)  # noqa: E731
    A = sp.DeviceCSR(rows, cols, t(rp), t(ci), t(va))
    d_x = t(x)
    y_plain = plain_merge(sp, A, d_x, rows, cols)
    assert_within_tolerance(y_plain, y64, scale, f"{what} plain")
    for cap in caps:
        plan = sp.CsrPlan(A.ptr, cap, force=True)
        n_hot, hot_nnz, mode = plan.info()
        if expect_mode is not None:  # 1 / 2: hub-column kernel (table / whole x); 3 / 4: segmented stream
            assert mode == expect_mode + (2 if SEG else 0), (what, cap, n_hot, mode)
        mode = mode - 2 if mode >= 3 else mode
        if expect_mode == 1:
            assert n_hot > 0
        if mode == 1 and n_hot > 0:
            assert n_hot <= (cap if cap > 0 else 1 << 20) and 0 < hot_nnz <= len(ci)
            # the admitted columns are the most referenced ones
            counts = np.bincount(ci, minlength=cols)
            order = np.sort(counts)[::-1]
            assert hot_nnz == int(order[:n_hot].sum()), (what, cap, n_hot)
        d_y = torch.full((rows,), float("nan"), dtype=torch.float32, device=dev)
        assert plan.spmv(d_x, d_y) == 0
        torch.cuda.synchronize()
        y = d_y.cpu().numpy()
        d_y.fill_(float("nan"))
        assert plan.spmv(d_x, d_y) == 0  # the plan is reusable, and the result reproducible
        torch.cuda.synchronize()
        assert np.array_equal(bits(y), bits(d_y.cpu().numpy())), f"{what} cap {cap}: two products differ"
        assert_within_tolerance(y, y64, scale, f"{what} cap {cap}")
        if HUB:
            assert np.array_equal(bits(y), bits(y_plain)), f"{what} cap {cap}: differs from plain MERGE_PATH"
        plan.close()


@pytest.mark.parametrize("scale,ef,seed", [(12, 8, 2), (15, 16, 3), (17, 16, 4)])
def test_rmat_hub_table_matches_plain_merge_path(sp, orc, cuda, scale, ef, seed):
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, ef, seed, "cpu")
    x = gen.vector_pm1(n, seed + 50, "cpu").numpy()
    check_plan(sp, orc, cuda, n, n, rp.numpy(), ci.numpy(), va.numpy(), x, caps=(4, 64, 1000), what=f"rmat {scale}",
               expect_mode=1)
    # device maximum: at these sizes every column fits -> the table is x itself
    check_plan(sp, orc, cuda, n, n, rp.numpy(), ci.numpy(), va.numpy(), x, caps=(0,), what=f"rmat {scale} all",
               expect_mode=2 if n <= 40000 else 1)


@pytest.mark.parametrize("rows,cols,avg,skew,seed", [
    (1, 1, 1, 0.0, 1), (5000, 70000, 9, 0.3, 2), (70000, 70000, 3, 0.05, 3), (300, 100000, 700, 0.0, 4),
    (100003, 65537, 3, 0.0, 5), (20000, 20000, 40, 0.5, 6)])
def test_random_shapes(sp, orc, cuda, rows, cols, avg, skew, seed):
    gen = gen_mod()
    rp, ci, va = gen.random_csr(rows, cols, avg, seed, "cpu", skew)
    x = gen.vector_pm1(cols, seed + 100, "cpu").numpy()
    check_plan(sp, orc, cuda, rows, cols, rp.numpy(), ci.numpy(), va.numpy(), x, caps=(8, 512, 0),
               what=f"random {rows}x{cols}")


def test_tile_geometry_edge_cases(sp, orc, cuda):
    """Rows far longer than a tile (tiles without a single row end, 513 load groups when the span
    starts unaligned), empty rows before / between / after, nnz not a multiple of 4, a single row."""
    rng = np.random.default_rng(7)
    cols = 60000
    for lens in ([100001], [1, 50003, 0, 0, 50002], [0, 0, 70001, 0], [3, 90001, 1], [2047, 2049, 1, 4095],
                 [0] * 3000 + [7] + [0] * 3000, [5] * 10000):
        lens = np.array(lens)
        rp = np.zeros(len(lens) + 1, np.int32)
        rp[1:] = np.cumsum(lens)
        nnz = int(rp[-1])
        # hub-heavy columns: half of the entries fall on 32 columns
        hub = rng.integers(0, 32, nnz) * 1777
        cold = rng.integers(0, cols, nnz)
        ci = np.where(rng.random(nnz) < 0.5, hub, cold).astype(np.int32)
        for r in range(len(lens)):
            ci[rp[r]:rp[r + 1]].sort()
        va = rng.uniform(-1, 1, nnz).astype(np.float32)
        x = rng.uniform(-1, 1, cols).astype(np.float32)
        check_plan(sp, orc, cuda, len(lens), cols, rp, ci, va, x, caps=(16, 40), what=f"lens {lens[:5].tolist()}",
                   expect_mode=1 if nnz > 1000 else None)


def test_unaligned_values_pointer(sp, orc, cuda):
    gen = gen_mod()
    rows, cols = 30000, 80000
    rp, ci, va = gen.random_csr(rows, cols, 7, 31, "cpu", 0.2)
    x = gen.vector_pm1(cols, 32, "cpu")
    y64, scale = orc.spmv_csr_f64(rows, rp.numpy(), ci.numpy(), va.numpy(), x.numpy())
    pad = lambda t: torch.cat([torch.zeros(1, dtype=t.dtype), t]).to(cuda)[1:]  # noqa: E731
    d_rp, d_ci, d_va, d_x = pad(rp), pad(ci), pad(va), pad(x)
    A = sp.DeviceCSR(rows, cols, d_rp, d_ci, d_va)
    for cap in (100, 0):  # hub table with unaligned values; cap 0 -> device maximum
        plan = sp.CsrPlan(A.ptr, cap, force=True)
        d_y = torch.zeros(rows + 1, dtype=torch.float32, device=cuda)[1:]
        assert plan.spmv(d_x, d_y) == 0
        torch.cuda.synchronize()
        assert_within_tolerance(d_y.cpu().numpy(), y64, scale, f"unaligned cap {cap}")
        plan.close()


def test_values_are_read_live_and_plan_follows_uploads(sp, orc, cuda):
    """The plan re-encodes col_indices only: new values in the same pattern need no new plan."""
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(14, 16, 9, cuda)
    A = sp.DeviceCSR(n, n, rp, ci, va)
    x = gen.vector_pm1(n, 3, cuda)
    plan = sp.CsrPlan(A.ptr, 256, force=True)
    va.mul_(-2.5)
    y = torch.empty(n, device=cuda)
    assert plan.spmv(x, y) == 0
    y_plain = plain_merge(sp, A, x, n, n)
    y64, scale = orc.spmv_csr_f64(n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), x.cpu().numpy())
    assert_within_tolerance(y.cpu().numpy(), y64, scale, "new values, old plan")
    if HUB:
        assert np.array_equal(bits(y.cpu().numpy()), bits(y_plain))
    plan.close()


def test_pagerank_steps_with_and_without_a_plan(sp, orc, cuda):
    """The fused PageRank iteration through the planned kernels, stepped for a fixed iteration count by a
    loop written here: same ranks (L1 <= 1e-6 against the f64 restatement of the reference recurrence,
    src/pagerank.cu:93-150) and the same residuals as through the plain tile kernel.  The whole graph on
    one GPU takes the segmented stream (different, fixed summation order); a ROW SHARD takes the
    hub-column kernel, whose r_new slice must equal the plain tile kernel's bit for bit (only the source
    of x[col] changes)."""
    gen = gen_mod()
    import gpu_spmv_b200.dist as D
    n, rp, ci, va = gen.rmat_pagerank_csr(16, 16, 11, cuda)
    iters = 12
    outs = []
    for cap in (0, 300, -1):
        shard = D.CudaShard(n, 0, rp, ci, va)
        used = shard.set_hot(cap, force=True)
        assert (used == 0) == (cap == 0)
        shard.setup_dangling()
        r_old, r_new = torch.empty(n, device=cuda), torch.empty(n, device=cuda)
        partial = torch.zeros(3, dtype=torch.float64, device=cuda)
        shard.init_vector(r_old)
        for _ in range(iters):
            shard(r_old, r_new, partial)
            shard.dsum.copy_(partial[2:3].to(torch.float32))  # the dangling mass of the vector just written
            r_old, r_new = r_new, r_old
        l2, l1 = partial[:2].tolist()
        outs.append((shard.normalize(r_old).cpu().numpy(), float(np.sqrt(np.float32(l2))), l1))
        shard.close()
    o_ranks, _, o_l2, o_l1, _ = orc.pagerank_f64(n, n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), 0.85, 0.0,
                                                 iters, fixed_it=iters)
    for ranks, l2, l1 in outs:
        assert np.abs(ranks.astype(np.float64) - o_ranks).sum() <= 1e-6
        assert abs(l2 - o_l2) <= 1e-8 + 1e-3 * o_l2 and abs(l1 - o_l1) <= 1e-8 + 1e-3 * o_l1
    for ranks, _, _ in outs[1:]:
        assert np.abs(ranks.astype(np.float64) - outs[0][0]).sum() <= 1e-6

    # one step on a row shard (rows [lo, hi) of the graph): hub-column kernel against the plain tile kernel
    lo, hi = n // 5, (3 * n) // 4
    srp, sci, sva = D.extract_shard(rp, ci, va, lo, hi)
    shard = D.CudaShard(n, lo, srp, sci, sva)
    shard.setup_dangling()
    r_old = torch.empty(n, device=cuda)
    shard.init_vector(r_old)
    r_old.mul_(gen.vector_pm1(n, 2, cuda).abs() + 0.5)  # not the uniform start vector
    slices, partials = [], []
    for cap in (0, 300):
        used = shard.set_hot(cap, force=True)
        assert (used == 0) == (cap == 0)
        r_new = torch.full((n,), float("nan"), device=cuda)
        partial = torch.zeros(3, dtype=torch.float64, device=cuda)
        shard(r_old, r_new, partial)
        torch.cuda.synchronize()
        assert bool(torch.isnan(r_new[:lo]).all()) and bool(torch.isnan(r_new[hi:]).all())  # only the shard's rows
        slices.append(r_new[lo:hi].clone())
        partials.append(partial.cpu().numpy())
    if not SEG:
        assert torch.equal(slices[0].view(torch.int32), slices[1].view(torch.int32))
    assert float((slices[0] - slices[1]).abs().sum()) <= 1e-6
    assert np.allclose(partials[0], partials[1], rtol=1e-4 if SEG else 1e-9, atol=1e-18)
    shard.close()


def test_spmv_csr_attaches_a_plan_to_csr_to_gpu_uploads(sp, orc, cuda):
    """Drop-in path with automatic plans switched ON (they are opt-in: off by default, a drop-in must
    not cache the sparsity pattern behind the caller's back): spmv_csr(MERGE_PATH) on arrays uploaded
    by csr_to_gpu builds the plan on the second call (large scale-free matrix), later calls run the
    hub-table kernel with identical results; csr_forget_plan / csr_free_gpu drop it."""
    from gpu_helpers import GpuCSR, run_csr
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(19, 16, 21, "cpu")
    x = gen.vector_pm1(n, 5, "cpu").numpy()
    A = GpuCSR(sp, n, n, rp.numpy(), ci.numpy(), va.numpy())
    y64, scale = orc.spmv_csr_f64(n, A.rp, A.ci, A.va, x)
    assert sp.lib.spmv_b200_auto_plan_enabled() == 0  # default: off
    for _ in range(3):
        y0, _ = run_csr(sp, A.mat, x, MERGE, cuda, n)
        assert sp.csr_auto_plan_info(A.mat) == (0, 0)
    sp.lib.spmv_b200_set_auto_plan(1)
    y1, _ = run_csr(sp, A.mat, x, MERGE, cuda, n)
    assert sp.csr_auto_plan_info(A.mat) == (0, 0)
    y2, _ = run_csr(sp, A.mat, x, MERGE, cuda, n)
    hot_columns, hot_nnz = sp.csr_auto_plan_info(A.mat)
    assert hot_columns > 0 and hot_nnz * 8 >= len(A.ci)
    y3, res = run_csr(sp, A.mat, x, MERGE, cuda, n)
    assert_within_tolerance(y1, y64, scale, "first call")
    assert_within_tolerance(y2, y64, scale, "second call (planned)")
    assert np.array_equal(bits(y2), bits(y3))
    assert res.elapsed_ms > 0
    sp.csr_forget_plan(A.mat)
    assert sp.csr_auto_plan_info(A.mat) == (0, 0)
    y4, _ = run_csr(sp, A.mat, x, MERGE, cuda, n)
    assert np.array_equal(bits(y1), bits(y4)) and np.array_equal(bits(y0), bits(y1))
    sp.lib.spmv_b200_set_auto_plan(0)
    A.close()


def test_plan_kind_follows_the_measured_structure(sp, orc, cuda):
    """A scale-free matrix gets the hub-column kernel, a regular one with >= 4 non-zeros per row the
    segmented-stream kernel (no hub worth a table), both through the same CsrPlan call."""
    if SEG:
        pytest.skip("SPMV_B200_PLAN forces one kernel")
    gen = gen_mod()
    rp, ci, va = gen.laplacian_2d_csr(1500, cuda)
    n = 1500 * 1500
    A = sp.DeviceCSR(n, n, rp, ci, va)
    x = gen.vector_pm1(n, 3, cuda)
    plan = sp.CsrPlan(A.ptr)
    assert plan.info()[2] == 3
    y = torch.full((n,), float("nan"), device=cuda)
    assert plan.spmv(x, y) == 0
    torch.cuda.synchronize()
    y64, scale = orc.spmv_csr_f64(n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), x.cpu().numpy())
    assert_within_tolerance(y.cpu().numpy(), y64, scale, "laplacian through the segmented-stream plan")
    plan.close()
    n2, rp2, ci2, va2 = gen.rmat_pagerank_csr(19, 16, 5, cuda)
    A2 = sp.DeviceCSR(n2, n2, rp2, ci2, va2)
    plan2 = sp.CsrPlan(A2.ptr)
    assert plan2.info()[2] == 1
    plan2.close()


def test_whole_file_with_segmented_stream_forced(cuda):
    """The whole file again with SPMV_B200_PLAN=seg (read once per process, hence the subprocess)."""
    if SEG:
        pytest.skip("already forced")
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_hot.py"), "-q", "-x", "-m", "gpu"]
    p = subprocess.run(cmd, env={**os.environ, "SPMV_B200_PLAN": "seg"}, cwd=root, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout[-3000:]


def test_full_size_rmat24_properties(sp, cuda):
    """BASELINE config 4 at full size (R-MAT scale 24, 268 M non-zeros), size-independent properties.
    The f64 oracle is too slow here, so the checks are relative to SCALAR_CSR (sequential per-row
    order == spmv_cpu_csr, proven bit-exact at oracle sizes in test_gpu_spmv.py) with the north_star
    row scale sum_j |a_ij x_j| computed by a product over |A|, |x|:
      * MERGE_PATH and both planned kernels within 1e-5 * scale of it, row by row;
      * the hub-column plan BIT-IDENTICAL to MERGE_PATH (only the source of x[col] changes);
      * linearity A(2x) = 2 A x exactly for every kernel (power-of-two scaling is exact in fp32);
      * rows without non-zeros are exactly 0."""
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(24, 16, 44, cuda)
    assert ci.numel() == 268435456
    A = sp.DeviceCSR(n, n, rp, ci, va)
    x = gen.vector_pm1(n, 11, cuda)
    y_sc, y_mg, y_p, scale = (torch.empty(n, device=cuda) for _ in range(4))
    assert sp.spmv_csr(A.ptr, x, y_sc, sp.make_config(sp.SCALAR_CSR), n).error_code == 0
    assert sp.spmv_csr(A.ptr, x, y_mg, sp.make_config(sp.MERGE_PATH), n).error_code == 0
    absA = sp.DeviceCSR(n, n, rp, ci, va.abs())
    assert sp.spmv_csr(absA.ptr, x.abs(), scale, sp.make_config(sp.SCALAR_CSR), n).error_code == 0
    assert bool(((y_mg - y_sc).abs() <= 1e-5 * scale).all())
    empty = (rp[1:] == rp[:-1])
    assert int(empty.sum()) > 0 and bool((y_mg[empty] == 0).all())
    plan = sp.CsrPlan(A.ptr)  # scale-free: the hub-column kernel (the segmented stream under SPMV_B200_PLAN=seg)
    assert plan.info()[2] == (3 if SEG else 1) and plan.info()[0] > 0
    y_p.fill_(float("nan"))
    assert plan.spmv(x, y_p) == 0
    torch.cuda.synchronize()
    assert bool(((y_p - y_sc).abs() <= 1e-5 * scale).all()) and bool((y_p[empty] == 0).all())
    if not SEG:
        assert torch.equal(y_p.view(torch.int32), y_mg.view(torch.int32))
    y2 = torch.empty(n, device=cuda)
    assert plan.spmv(x * 2, y2) == 0
    torch.cuda.synchronize()
    assert torch.equal(y2, y_p * 2)
    plan.close()


def test_snapshot_plan_routes_uniform_matrices_to_ell(sp, orc, cuda):
    """SPMV_B200_PLAN_SNAPSHOT_VALUES: a uniform matrix is re-laid out as ELL inside the plan (the
    routing the reference's ELL_KERNEL enumerator promises, spmv.h:16).  The ELL kernel keeps the CSR
    order inside a row, so the result is BIT-IDENTICAL to spmv_cpu_csr; new values need
    refresh_values(); a skewed matrix ignores the flag."""
    gen = gen_mod()
    grid = 700
    n = grid * grid
    rp, ci, va = gen.laplacian_2d_csr(grid, cuda)
    A = sp.DeviceCSR(n, n, rp, ci, va)
    x = gen.vector_pm1(n, 8, cuda)
    plan = sp.CsrPlan(A.ptr, snapshot_values=True)
    assert plan.info()[2] == 5
    y = torch.full((n,), float("nan"), device=cuda)
    assert plan.spmv(x, y) == 0
    torch.cuda.synchronize()
    expect = orc.spmv_csr(n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), x.cpu().numpy())
    assert np.array_equal(bits(y.cpu().numpy()), bits(expect))
    va.mul_(1.5).add_(0.25)  # same pattern, new values
    assert plan.spmv(x, y) == 0
    torch.cuda.synchronize()
    assert np.array_equal(bits(y.cpu().numpy()), bits(expect))  # the snapshot is still the old one
    assert plan.refresh_values() == 0
    assert plan.spmv(x, y) == 0
    torch.cuda.synchronize()
    expect2 = orc.spmv_csr(n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), x.cpu().numpy())
    assert np.array_equal(bits(y.cpu().numpy()), bits(expect2)) and not np.array_equal(bits(expect), bits(expect2))
    plan.close()
    # without the flag the same matrix takes a kernel that reads the values live
    live = sp.CsrPlan(A.ptr, force=True)
    assert live.info()[2] in (0, 3)
    live.close()
    # a skewed matrix is not ELL material: the flag changes nothing
    n2, rp2, ci2, va2 = gen.rmat_pagerank_csr(14, 16, 3, cuda)
    A2 = sp.DeviceCSR(n2, n2, rp2, ci2, va2)
    p2 = sp.CsrPlan(A2.ptr, 64, force=True, snapshot_values=True)
    assert p2.info()[2] in (1, 3)
    p2.close()
