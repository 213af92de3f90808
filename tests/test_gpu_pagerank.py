"""Parity of the fused PageRank iteration with the reference recurrence
(src/pagerank.cu:50-153) through the C ABI.  north_star: rank vectors within
an L1 distance of 1e-6, identical top-k up to ties."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def gen_mod():
    import gpu_spmv_b200.gen as gen
    return gen


def gpu_pagerank(sp, n, rp, ci, va, damping=0.85, tol=1e-6, max_it=100):
    G = sp.csr_from_arrays(n, n, rp, ci, va)
    assert sp.csr_to_gpu(G) == 0
    res, ranks = sp.pagerank(G, sp.make_pagerank_config(damping, tol, max_it))
    out = (ranks, res.iterations, res.final_residual, bool(res.converged))
    sp.pagerank_free(res)
    assert not res.ranks  # pagerank_free nulls the pointer and is idempotent
    sp.pagerank_free(res)
    sp.csr_destroy(G)
    return out


def same_top_k_up_to_ties(ranks_a, ranks_b, k, tol=1e-7):
    """Top-k sets may differ only in members whose ranks are within tol of the k-th rank."""
    k = min(k, len(ranks_a))
    top_a, top_b = np.argsort(-ranks_a, kind="stable")[:k], np.argsort(-ranks_b, kind="stable")[:k]
    kth = ranks_a[top_a[-1]]
    for i in set(top_a.tolist()) ^ set(top_b.tolist()):
        assert abs(ranks_a[i] - kth) <= tol and abs(ranks_b[i] - kth) <= tol, i
    assert np.all(np.abs(np.sort(ranks_a[top_a]) - np.sort(ranks_b[top_b])) <= tol)


def test_reference_property_inputs(sp, orc, cuda, golden):
    """Inputs of PageRankPropertyTest.ScoreInvariants (tests/test_pagerank.cu:18-77): the
    reference's invariants, then the values against the literal fp32 restatement."""
    g = golden.pr
    for it in range(int(g["n_cases"][0])):
        p = f"p{it}_"
        n = int(g[p + "n"][0])
        rp, ci, va = g[p + "row_ptrs"], g[p + "col_indices"], g[p + "values"]
        ranks, iters, res, conv = gpu_pagerank(sp, n, rp, ci, va, 0.85, 1e-5, 50)
        assert np.all(ranks >= 0) and abs(float(ranks.sum(dtype=np.float64)) - 1.0) < 1e-4
        assert conv or iters == 50
        if conv:
            assert res < 1e-5
        o_ranks, o_it, o_res, o_conv = orc.pagerank_f32(n, n, rp, ci, va, 0.85, 1e-5, 50)
        assert abs(iters - o_it) <= 1 and conv == o_conv
        o_same, _, _, _, _ = orc.pagerank_f64(n, n, rp, ci, va, 0.85, 1e-5, 50, fixed_it=iters)
        assert np.abs(ranks.astype(np.float64) - o_same).sum() <= 1e-6
        assert np.abs(ranks.astype(np.float64) - o_ranks).sum() <= 1e-5  # <= one iteration apart near the threshold
        same_top_k_up_to_ties(ranks, o_same, 5)


def test_reference_unit_cases(sp, orc, cuda):
    # 3-cycle (tests/test_pagerank.cu:140-164): converged, equal ranks
    rp, ci, va = orc.csr_from_dense(np.array([[0, 0, 1], [1, 0, 0], [0, 1, 0]], np.float32))
    ranks, iters, res, conv = gpu_pagerank(sp, 3, rp, ci, va)
    assert conv and np.allclose(ranks, 1 / 3, atol=1e-4)
    # 4-node symmetric graph, top-2 (tests/test_pagerank.cu:166-189)
    adj = np.array([[0, 1, 1, 0], [1, 0, 1, 1], [1, 1, 0, 1], [0, 1, 1, 0]], np.float32)
    adj = adj / adj.sum(axis=0, keepdims=True)
    rp, ci, va = orc.csr_from_dense(adj)
    ranks, _, _, _ = gpu_pagerank(sp, 4, rp, ci, va)
    ids, vals = sp.pagerank_top_k(ranks, 2)
    assert set(ids.tolist()) == {1, 2} and vals[0] >= vals[1]
    # graph with dangling nodes and isolated rows; not on the device -> normalised initial vector (src/pagerank.cu:105-107)
    G = sp.csr_from_arrays(3, 3, rp[:4] * 0, [], [])
    res, r = sp.pagerank(G, None)
    assert res.iterations == 0 and not res.converged and np.allclose(r, 1 / 3)
    sp.pagerank_free(res)
    sp.csr_destroy(G)
    res, r = sp.pagerank(None, None)
    assert r is None and res.iterations == 0


def gpu_pagerank_device(sp, n, rp, ci, va, cuda, damping=0.85, tol=1e-6, max_it=100):
    """The device-resident entry point: f64 accumulators for every global sum, f64 normalisation."""
    G = sp.DeviceCSR(n, n, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    d_ranks = torch.empty(n, device=cuda)
    rc, iters, res, conv, l1 = sp.pagerank_device(G.ptr, d_ranks, sp.make_pagerank_config(damping, tol, max_it))
    assert rc == 0
    return d_ranks.cpu().numpy(), iters, res, conv, l1


@pytest.mark.parametrize("scale,edge_factor,seed", [(8, 4, 1), (12, 8, 2), (15, 16, 3), (17, 16, 4)])
def test_rmat_graphs_vs_restatement(sp, orc, cuda, scale, edge_factor, seed):
    """R-MAT graphs (dangling nodes, empty rows, hub rows spanning many merge tiles).

    Two oracles, two entry points (DESIGN.md, "PageRank numerics"):
      * pagerank_device (f64 accumulators everywhere) vs the f64-accumulator restatement: L1 <= 1e-6
        at every size -- this is the recurrence evaluated accurately.
      * pagerank() (drop-in API; final normalisation is the reference's own sequential fp32 host
        sum) vs the LITERAL fp32 restatement: L1 <= 2e-6 where the reference's fp32 sums are
        still accurate (n <= 2^13).  Beyond that the literal reference drifts from the exact
        recurrence by itself (measured below: ~1e-3 in L1 at n = 2^17), so we only require that we
        are no further from it than it is from the exact recurrence."""
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, edge_factor, seed, "cpu")
    rp, ci, va = rp.numpy(), ci.numpy(), va.numpy()
    n_dangling, _ = orc.find_dangling(n, n, rp, ci, va)
    assert n_dangling > 0

    d_ranks, iters, res, conv, l1 = gpu_pagerank_device(sp, n, rp, ci, va, cuda)
    assert conv and res < 1e-6
    o_ranks, o_it, o_l2, o_l1, o_conv = orc.pagerank_f64(n, n, rp, ci, va, 0.85, 1e-6, 100)
    assert abs(iters - o_it) <= 1
    o_same, _, l2_same, l1_same, _ = orc.pagerank_f64(n, n, rp, ci, va, 0.85, 1e-6, 100, fixed_it=iters)
    assert np.abs(d_ranks.astype(np.float64) - o_same).sum() <= 1e-6
    assert abs(res - l2_same) <= 1e-8 + 1e-3 * l2_same and abs(l1 - l1_same) <= 1e-8 + 1e-3 * l1_same
    assert abs(float(d_ranks.sum(dtype=np.float64)) - 1.0) < 1e-6
    same_top_k_up_to_ties(d_ranks, o_same, 20)

    ranks, a_iters, a_res, a_conv = gpu_pagerank(sp, n, rp, ci, va, 0.85, 1e-6, 100)
    assert (a_iters, a_conv) == (iters, conv)
    l_ranks, l_it, l_res, l_conv = orc.pagerank_f32(n, n, rp, ci, va, 0.85, 1e-6, 100)
    assert abs(l_it - a_iters) <= 1
    ours_vs_literal = np.abs(ranks.astype(np.float64) - l_ranks).sum()
    literal_vs_exact = np.abs(l_ranks.astype(np.float64) - o_ranks).sum()
    print(f"scale {scale}: |ours - literal fp32 reference|_1 = {ours_vs_literal:.3e}; "
          f"|literal fp32 reference - f64 recurrence|_1 = {literal_vs_exact:.3e}")
    if n <= 1 << 13:
        assert ours_vs_literal <= 2e-6
        same_top_k_up_to_ties(ranks, l_ranks, 20, tol=2e-7)
    else:
        assert ours_vs_literal <= literal_vs_exact + 1e-6


def test_device_resident_api_and_shards_on_one_gpu(sp, orc, cuda):
    """spmv_b200_pagerank_device and the sharded building blocks: three row shards stepped
    one after another on one GPU must reproduce the unsharded iteration."""
    gen = gen_mod()
    import gpu_spmv_b200.dist as D
    n, rp, ci, va = gen.rmat_pagerank_csr(14, 16, 5, cuda)
    G = sp.DeviceCSR(n, n, rp, ci, va)
    d_ranks = torch.empty(n, device=cuda)
    rc, iters, res, conv, l1 = sp.pagerank_device(G.ptr, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100))
    assert rc == 0 and conv and l1 > 0
    o_same, _, l2, o_l1, _ = orc.pagerank_f64(n, n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), 0.85, 1e-6,
                                               100, fixed_it=iters)
    assert np.abs(d_ranks.cpu().numpy().astype(np.float64) - o_same).sum() <= 1e-6
    assert abs(l1 - o_l1) <= 1e-3 * o_l1 + 1e-9

    bounds = D.partition_rows(rp, 3)
    assert bounds == D.partition_rows(rp.cpu(), 3) == orc.partition_rows(n, rp.cpu().numpy(), 3).tolist()
    shards = []
    for p in range(3):
        srp, sci, sva = D.extract_shard(rp, ci, va, bounds[p], bounds[p + 1])
        shards.append(D.CudaShard(n, bounds[p], srp, sci, sva))
    for s in shards:
        s.setup_dangling()
    # every shard contributes its own column sums; emulate the all-reduce by summing bits' sources
    colsum = torch.zeros(n, dtype=torch.float64, device=cuda)
    for s in shards:
        assert sp.lib.spmv_b200_pr_colsum(s.plan, sp.dptr(colsum), None) == 0
    for s in shards:
        assert sp.lib.spmv_b200_pr_dangling_bits(sp.dptr(colsum), n, sp.dptr(s.bits), None) == 0
    r_old, r_new = torch.empty(n, device=cuda), torch.empty(n, device=cuda)
    shards[0].init_vector(r_old)
    dsum0 = shards[0].dsum.clone()
    total = torch.zeros(3, dtype=torch.float64, device=cuda)
    part = torch.zeros(3, dtype=torch.float64, device=cuda)
    for it in range(iters):
        total.zero_()
        for s in shards:
            s.dsum.copy_(dsum0)
            s(r_old, r_new, part)
            total += part
        dsum0 = total[2:3].to(torch.float32)
        r_old, r_new = r_new, r_old
    final = shards[0].normalize(r_old)
    assert np.abs(final.cpu().numpy().astype(np.float64) - o_same).sum() <= 1e-6
    assert abs(float(torch.sqrt(total[0].float())) - res) <= 1e-3 * res + 1e-9
    for s in shards:
        s.close()


def test_pr_step_p2p_stores_the_shard_into_every_peer_buffer(sp, cuda):
    """spmv_b200_pr_step_p2p on one GPU, with a two-entry peer table whose other entry is a second buffer on
    the same device: the shard's rows must land in both buffers bit for bit as spmv_b200_pr_step writes them,
    with the same partial sums, and no row outside the shard may change.  A row shard through the plain tile
    kernel and the hub-column kernel, and the whole graph through the segmented stream."""
    gen = gen_mod()
    import gpu_spmv_b200.dist as D
    n, rp, ci, va = gen.rmat_pagerank_csr(14, 16, 5, cuda)
    shard_rows = (n // 5, (3 * n) // 4)
    for (lo, hi), cap in ((shard_rows, 0), (shard_rows, 300), ((0, n), -1)):
        srp, sci, sva = D.extract_shard(rp, ci, va, lo, hi)
        shard = D.CudaShard(n, lo, srp, sci, sva)
        assert (shard.set_hot(cap, force=True) == 0) == (cap == 0)
        shard.setup_dangling()
        r_old = torch.empty(n, device=cuda)
        shard.init_vector(r_old)
        r_old.mul_(gen.vector_pm1(n, 2, cuda).abs() + 0.5)  # not the uniform start vector
        ref = torch.full((n,), float("nan"), device=cuda)
        ref_partial = torch.zeros(3, dtype=torch.float64, device=cuda)
        shard(r_old, ref, ref_partial)
        torch.cuda.synchronize()
        for self_rank in (0, 1):
            mine = torch.full((n,), float("nan"), device=cuda)
            peer = torch.full((n,), -1.0, device=cuda)
            table = (C.c_void_p * 2)()
            table[self_rank], table[1 - self_rank] = mine.data_ptr(), peer.data_ptr()
            partial = torch.full((3,), float("nan"), dtype=torch.float64, device=cuda)
            rc = sp.lib.spmv_b200_pr_step_p2p(shard.plan, sp.dptr(r_old), sp.dptr(mine), shard.damping, sp.dptr(shard.dsum),
                                              sp.dptr(shard.bits), sp.dptr(partial), table, 2, self_rank, None)
            assert rc == 0, sp.spmv_error_string(rc)
            torch.cuda.synchronize()
            for out in (mine, peer):
                assert torch.equal(out[lo:hi].view(torch.int32), ref[lo:hi].view(torch.int32)), (cap, self_rank)
            assert torch.equal(partial, ref_partial), (cap, self_rank, partial, ref_partial)
            assert bool(torch.isnan(mine[:lo]).all()) and bool(torch.isnan(mine[hi:]).all())
            assert bool((peer[:lo] == -1.0).all()) and bool((peer[hi:] == -1.0).all())
        shard.close()


IPC_CHILD = """
import ctypes as C, sys
import torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from _load_pkg import load_pkg
sp = load_pkg()
import gpu_spmv_b200.dist as D
torch.cuda.set_device(0)
n = int(sys.argv[3])
ptr = C.c_void_p()
rc = sp.lib.spmv_b200_ipc_open(bytes.fromhex(sys.argv[2]), C.byref(ptr))
assert rc == 0, sp.spmv_error_string(rc)
got = D._tensor_from_ptr(ptr.value, n, torch.device("cuda:0")).cpu()
assert torch.equal(got, torch.arange(n, dtype=torch.float32) * 0.5 - 7.0), "the mapped buffer holds other values"
assert sp.lib.spmv_b200_ipc_close(ptr) == 0
print("IPC OK", flush=True)
"""


def test_ipc_buffer_mapped_by_a_child_process(sp, cuda):
    """spmv_b200_ipc_alloc / _open / _close / _free: a child process on the same GPU maps the buffer this process
    allocated, reads the pattern written here and closes its mapping; then this process frees the buffer."""
    import subprocess
    import sys
    import gpu_spmv_b200.dist as D
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 1 << 20
    ptr, handle = C.c_void_p(), C.create_string_buffer(64)
    assert sp.lib.spmv_b200_ipc_alloc(n * 4, C.byref(ptr), handle) == 0
    try:
        buf = D._tensor_from_ptr(ptr.value, n, cuda)
        buf.copy_(torch.arange(n, dtype=torch.float32, device=cuda) * 0.5 - 7.0)
        torch.cuda.synchronize()
        p = subprocess.run([sys.executable, "-c", IPC_CHILD, root, handle.raw.hex(), str(n)], cwd=root,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert p.returncode == 0 and "IPC OK" in p.stdout, p.stdout[-4000:]
    finally:
        assert sp.lib.spmv_b200_ipc_free(ptr) == 0


def test_reference_cuda_pagerank_agrees(sp, orc, ref, cuda):
    """Secondary oracle: the reference's own pagerank() (GPU SpMV + host loops) compiled for
    sm_100a from the unmodified sources, where it is trustworthy (n <= 2^15)."""
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(13, 8, 6, "cpu")
    rp, ci, va = rp.numpy(), ci.numpy(), va.numpy()
    h, keep = ref.csr_wrap(n, n, rp, ci, va)
    assert ref.L.ref_csr_to_gpu(h) == 0
    r_ref = np.empty(n, np.float32)
    res, conv = C.c_float(0), C.c_int(0)
    it_ref = ref.L.ref_pagerank(h, 0.85, 1e-6, 100, r_ref.ctypes.data_as(C.POINTER(C.c_float)), C.byref(res),
                                C.byref(conv))
    ranks, iters, my_res, my_conv = gpu_pagerank(sp, n, rp, ci, va)
    assert bool(conv.value) == my_conv and abs(it_ref - iters) <= 1
    assert np.abs(ranks.astype(np.float64) - r_ref).sum() <= 2e-6
    same_top_k_up_to_ties(ranks, r_ref, 10, tol=2e-7)
    ids, vals = sp.pagerank_top_k(ranks, 10)
    rid, rv = np.empty(10, np.int32), np.empty(10, np.float32)
    ref.L.ref_pagerank_top_k(ranks.ctypes.data_as(C.POINTER(C.c_float)), n, 10, rid.ctypes.data_as(C.POINTER(C.c_int)),
                             rv.ctypes.data_as(C.POINTER(C.c_float)))
    assert np.array_equal(vals, rv)  # same ranks position by position (ids may differ only on ties)


@pytest.mark.parametrize("n,k,kind", [(1, 1, "rand"), (10, 20, "rand"), (5000, 7, "rand"), (300000, 100, "rand"),
                                      (300000, 1000, "ties"), (70000, 50, "const"), (100003, 10, "neg")])
def test_device_top_k_matches_host_top_k(sp, cuda, n, k, kind):
    """spmv_b200_pagerank_top_k_device against the API's host pagerank_top_k (src/pagerank.cu:162-185):
    identical rank values position by position; node ids identical wherever ranks are distinct, and
    ascending inside a run of equal ranks (the reference leaves ties unordered)."""
    rng = np.random.default_rng(n + k)
    if kind == "rand":
        v = rng.random(n).astype(np.float32)
    elif kind == "ties":   # few distinct values: the threshold falls inside a long run of equal ranks
        v = (rng.integers(0, 12, n) / 16.0).astype(np.float32)
    elif kind == "const":
        v = np.full(n, 1.0 / n, np.float32)
    else:                  # negative values and zeros order correctly too
        v = rng.uniform(-1, 1, n).astype(np.float32)
        v[::7] = 0.0
    ids, vals = sp.pagerank_top_k_device(torch.as_tensor(v).to(cuda), k)
    h_ids, h_vals = sp.pagerank_top_k(v, k)
    kk = min(k, n)
    assert len(ids) == kk and np.array_equal(vals, h_vals)
    assert np.array_equal(v[ids], vals) and len(set(ids.tolist())) == kk
    expect = np.lexsort((np.arange(n), -v.astype(np.float64)))[:kk]  # rank descending, id ascending
    assert np.array_equal(ids, expect.astype(np.int32))


def test_residual_history(sp, orc, cuda):
    """spmv_b200_pagerank_device_history: the residual of every iteration is the one the stop rule saw
    (last entry == final_residual < tolerance, earlier ones above it, nothing written past the last iteration)
    and matches the f64 restatement of the recurrence run for the same number of iterations."""
    gen = gen_mod()
    n, rp, ci, va = gen.rmat_pagerank_csr(13, 8, 21, cuda)
    G = sp.DeviceCSR(n, n, rp, ci, va)
    d_ranks = torch.empty(n, device=cuda)
    rc, iters, res, conv, hist = sp.pagerank_device_history(G.ptr, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100), 64)
    assert rc == 0 and conv and 1 < iters <= 64
    assert np.all(np.isfinite(hist[:iters])) and np.all(np.isnan(hist[iters:]))
    assert hist[iters - 1] == np.float32(res) and res < 1e-6 and np.all(hist[:iters - 1] >= 1e-6)
    assert hist[iters - 1] < hist[0]
    for k in (1, iters // 2, iters):
        _, _, l2, _, _ = orc.pagerank_f64(n, n, rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(), 0.85, 1e-6, 100,
                                          fixed_it=k)
        assert abs(hist[k - 1] - l2) <= 1e-8 + 1e-3 * l2
    # a capacity shorter than the run keeps the first entries only
    rc, iters2, _, _, short = sp.pagerank_device_history(G.ptr, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100), 3)
    assert rc == 0 and iters2 == iters and np.array_equal(short, hist[:3])


def test_non_square_adjacency_is_rejected(sp, ref, cuda):
    """A matrix with num_cols != num_rows: the reference's first spmv_csr(adj, ..., vec_size = n) returns
    INVALID_DIMENSION, the loop breaks and pagerank() hands back the uniform vector with iterations = 0
    (src/pagerank.cu:102-107, :135-150).  The device entry points must reject it instead of gathering
    past the rank vector (ADVICE r1)."""
    gen = gen_mod()
    rows, cols = 64, 96
    rp, ci, va = gen.random_csr(rows, cols, 4, seed=8, device="cpu")
    rp, ci, va = rp.numpy(), ci.numpy(), va.numpy()
    G = sp.csr_from_arrays(rows, cols, rp, ci, va)
    assert sp.csr_to_gpu(G) == 0
    res, ranks = sp.pagerank(G, sp.make_pagerank_config(0.85, 1e-6, 50))
    assert res.iterations == 0 and not res.converged
    assert np.allclose(ranks, 1.0 / rows, rtol=1e-6)
    sp.pagerank_free(res)
    d_ranks = torch.empty(rows, device=cuda)
    rc = sp.pagerank_device(G, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 50))[0]
    assert rc == sp.SpMVError.INVALID_DIMENSION
    handle = C.c_void_p()
    assert sp.lib.spmv_b200_pr_plan_create(G, 0, rows, None, C.byref(handle)) == sp.SpMVError.INVALID_DIMENSION
    # the reference library itself (oracle/_ref: GPU SpMV + host loops) behaves the same way
    h, keep = ref.csr_wrap(rows, cols, rp, ci, va)
    assert ref.L.ref_csr_to_gpu(h) == 0
    r_ref = np.empty(rows, np.float32)
    r_res, r_conv = C.c_float(0), C.c_int(0)
    it_ref = ref.L.ref_pagerank(h, 0.85, 1e-6, 50, r_ref.ctypes.data_as(C.POINTER(C.c_float)), C.byref(r_res), C.byref(r_conv))
    assert it_ref == 0 and not r_conv.value and np.array_equal(r_ref, ranks)
    sp.csr_destroy(G)


def test_one_kernel_loop_for_small_graphs(sp, orc, cuda):
    """pagerank_small.cu: graphs of launch-bound size run the whole loop in one persistent cooperative kernel (grid
    barrier per iteration, stop rule on the device).  Same contract as the multi-kernel loop: within L1 1e-6 of the f64
    restatement at the same iteration count, the reference's stop rule (converged at the iteration the oracle converges,
    +-1 for a residual at the tolerance), residual history, max_iterations = 0 returns the initial vector; and the two
    loops agree with each other (child processes: the switch is read once per process)."""
    import subprocess
    import sys
    gen = gen_mod()
    for scale, ef, seed in ((6, 4, 3), (11, 16, 4), (15, 8, 5)):
        n, rp, ci, va = gen.rmat_pagerank_csr(scale, ef, seed, "cpu")
        rp_n, ci_n, va_n = rp.numpy(), ci.numpy(), va.numpy()
        G = sp.csr_from_arrays(n, n, rp_n, ci_n, va_n)
        assert sp.csr_to_gpu(G) == 0
        d_ranks = torch.empty(n, dtype=torch.float32, device=cuda)
        rc, iters, res, conv, l1 = sp.pagerank_device(G, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100))
        assert rc == 0 and conv and 1 <= iters <= 100 and res < 1e-6
        o_ranks, o_it, o_l2, o_l1, o_conv = orc.pagerank_f64(n, n, rp_n, ci_n, va_n, 0.85, 1e-6, 100, fixed_it=iters)
        assert np.abs(d_ranks.cpu().numpy().astype(np.float64) - o_ranks).sum() <= 1e-6, scale
        free_it = orc.pagerank_f64(n, n, rp_n, ci_n, va_n, 0.85, 1e-6, 100)[1]
        assert abs(free_it - iters) <= 1, (scale, free_it, iters)
        assert abs(float(d_ranks.double().sum()) - 1.0) <= 1e-5
        rc, it0, _, conv0, _ = sp.pagerank_device(G, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 0))
        assert rc == 0 and it0 == 0 and not conv0
        assert np.allclose(d_ranks.cpu().numpy(), 1.0 / n, rtol=1e-6, atol=0.0)
        rc, it_h, res_h, conv_h, hist = sp.pagerank_device_history(G, d_ranks, sp.make_pagerank_config(0.85, 1e-6, 100), capacity=100)
        assert rc == 0 and it_h == iters and conv_h and hist[iters - 1] == np.float32(res_h) and np.all(hist[:iters] > 0)
        assert np.all(np.isnan(hist[iters:]))
        sp.csr_destroy(G)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "scripts", "time_small_pagerank.py")], cwd=root, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:]
    print(p.stdout)
    dists = [float(ln.split("iterations ")[1].split(",")[0]) for ln in p.stdout.splitlines() if ln.startswith("scale ") and "L1 distance" in ln]
    assert len(dists) == 7 and max(dists) <= 1e-6, p.stdout[-2000:]
