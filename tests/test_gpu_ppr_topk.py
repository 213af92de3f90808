"""Per-seed top-K personalized PageRank (libspmv_b200_ppr_topk.so).

- Row c is the top of column c of the dense batch (spmv_b200_pagerank_personalized_batch), bit for bit, in the order
  rank descending, node id ascending; it equals pagerank_top_k_device of that column; places past n are (-1, 0.0);
  iterations, residuals, convergence and history are the batch's.
- Ties across the threshold are filled in ascending node order.
- A row does not depend on the batch (alone, at another position, in a later chunk, in a second run).
- k past the device memory for a dense n x k output runs and matches the dense batch on those seeds alone.
- The library ships exactly the kernels a call launches, none of libspmv_b200.so's, and exports exactly its header.
- Input validation needs no GPU and launches nothing; importing the package does not load the library."""
import ctypes as C
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from test_gpu_pagerank_batch import GRAPH_NAMES, _columns, _device_graph, _graphs
from test_gpu_pagerank_personalized import _sass_summary, graph, rmat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "gpu-spmv_b200", "lib")
D = 0.85


def _call(sp, A, k, offsets, nodes, weights, cfg, top, d_ids, d_vals, capacity=0):
    """The C entry point with raw arrays -> (rc, iterations, residual, converged, history)."""
    ip, fp = C.POINTER(C.c_int), C.POINTER(C.c_float)
    kk = max(k, 1)
    it, res, conv = np.zeros(kk, np.int32), np.zeros(kk, np.float32), np.zeros(kk, np.bool_)
    hist = np.full(kk * max(capacity, 1), np.nan, np.float32)
    arr = lambda a, t, p: np.ascontiguousarray(a, t).ctypes.data_as(p) if a is not None else None  # noqa: E731
    rc = sp.ppr_topk_lib().spmv_b200_pagerank_personalized_batch_top_k(
        A, C.byref(cfg) if cfg is not None else None, k, arr(offsets, np.int32, ip), arr(nodes, np.int32, ip),
        arr(weights, np.float32, fp), top, d_ids, d_vals, it.ctypes.data_as(ip), res.ctypes.data_as(fp),
        conv.ctypes.data_as(C.POINTER(C.c_bool)), hist.ctypes.data_as(fp) if capacity > 0 else None, capacity)
    return rc, it, res, conv, hist


def _counters(sp):
    return sp.launch_count(), sp.ppr_lib().spmv_b200_ppr_launch_count(), sp.ppr_topk_lib().spmv_b200_ppr_topk_launch_count()


# -------------------------------------------------------------------------------- input validation (CPU) ----
def test_rejected_inputs_launch_nothing(sp):
    """Every malformed call is INVALID_ARGUMENT before any device work.  The CSR has host arrays only and d_ids /
    d_vals are bogus non-NULL addresses: nothing could run anyway, and no library's launch counter moves."""
    bad_arg = int(sp.SpMVError.INVALID_ARGUMENT)
    n = 4
    A = sp.csr_create(0, 0, 0)
    sp.csr_from_dense(A, np.eye(n, dtype=np.float32), n, n)
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    fi, fv = C.c_void_p(0x1000), C.c_void_p(0x2000)
    cases = {
        "k = 0": (0, [0], [], None),
        "k < 0": (-1, [0], [], None),
        "offsets[0] != 0": (1, [1, 2], [0, 1], None),
        "decreasing offsets": (2, [0, 2, 1], [0, 1], None),
        "node < 0": (1, [0, 1], [-1], None),
        "node >= n": (1, [0, 1], [n], None),
        "repeated node": (1, [0, 2], [1, 1], None),
        "out of order": (1, [0, 2], [2, 1], None),
        "NaN weight": (1, [0, 2], [0, 1], [1.0, np.nan]),
        "+Inf weight": (1, [0, 1], [0], [np.inf]),
        "-Inf weight": (1, [0, 2], [0, 3], [1.0, -np.inf]),
        "negative weight": (2, [0, 1, 2], [0, 2], [1.0, -1e-30]),
        "zero column": (2, [0, 1, 2], [0, 3], [1.0, 0.0]),
        "empty column": (2, [0, 1, 1], [2], None),
        "nodes NULL": (1, [0, 1], None, None),
    }
    before = _counters(sp)
    for name, (k, off, nodes, w) in cases.items():
        assert _call(sp, A, k, off, nodes, w, cfg, 3, fi, fv)[0] == bad_arg, name
    good = ([0, 1, 3], [2, 0, 3], [1.0, 2.0, 0.5])
    assert _call(sp, None, 2, *good, cfg, 3, fi, fv)[0] == bad_arg  # NULL adjacency
    assert _call(sp, None, 2, None, None, None, cfg, 3, fi, fv)[0] == bad_arg  # NULL offsets
    for top in (0, -1, 1025):
        assert _call(sp, A, 2, *good, cfg, top, fi, fv)[0] == bad_arg, top
    assert _call(sp, A, 2, *good, cfg, 3, None, fv)[0] == bad_arg  # NULL d_ids
    assert _call(sp, A, 2, *good, cfg, 3, fi, None)[0] == bad_arg  # NULL d_vals
    f = sp.ppr_topk_lib().spmv_b200_pagerank_personalized_batch_top_k
    off, nod = np.array(good[0], np.int32), np.array(good[1], np.int32)
    ip = C.POINTER(C.c_int)
    it, res, conv = np.zeros(2, np.int32), np.zeros(2, np.float32), np.zeros(2, np.bool_)
    args = [off.ctypes.data_as(ip), nod.ctypes.data_as(ip), None, 3, fi, fv]
    outs = [it.ctypes.data_as(ip), res.ctypes.data_as(C.POINTER(C.c_float)), conv.ctypes.data_as(C.POINTER(C.c_bool))]
    for i in range(3):  # each NULL result array
        o = list(outs)
        o[i] = None
        assert f(A, C.byref(cfg), 2, *args, *o, None, 0) == bad_arg, i
    assert f(A, C.byref(cfg), 2, *args, *outs, None, 4) == bad_arg  # history capacity without a history array
    assert f(A, C.byref(cfg), 2, *args, *outs, None, -1) == bad_arg
    Z = sp.csr_create(0, 0, 0)  # n = 0: every column is necessarily empty
    assert _call(sp, Z, 1, [0, 0], [], None, cfg, 3, fi, fv)[0] == bad_arg
    assert _call(sp, Z, 1, [0, 1], [0], None, cfg, 3, fi, fv)[0] == bad_arg
    assert _counters(sp) == before
    sp.csr_destroy(A)
    sp.csr_destroy(Z)


def test_library_exports_exactly_its_header(sp):
    sp.ppr_topk_lib()  # built and loadable
    header = open(os.path.join(ROOT, "include", "spmv_b200_ppr_topk.h")).read()
    declared = set(re.findall(r"SPMV_B200_API[^;(]*?\b(spmv_b200_\w+)\s*\(", header))
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(LIBDIR, "libspmv_b200_ppr_topk.so")],
                         capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if line.split() and line.split()[-2] in "TtWwDdBbRrVvi"}
    assert declared == {"spmv_b200_pagerank_personalized_batch_top_k", "spmv_b200_ppr_topk_launch_count"}
    assert exported == declared


# --------------------------------------------------------------------------------------------- helpers ----
def _expected_row(col, top):
    """The first min(top, n) entries of a dense column by (rank descending, id ascending), padded to top."""
    n = col.size
    order = np.lexsort((np.arange(n), -col))[:min(top, n)]
    ids = np.full(top, -1, np.int32)
    vals = np.zeros(top, np.float32)
    ids[:order.size] = order
    vals[:order.size] = col[order]
    return ids, vals


def _assert_row(ids, vals, col, top, what):
    e_ids, e_vals = _expected_row(col, top)
    assert np.array_equal(ids, e_ids), f"{what}: ids {ids[:8]} vs {e_ids[:8]}"
    assert np.array_equal(vals.view(np.uint32), e_vals.view(np.uint32)), f"{what}: values differ"


def _bits(t):
    return t.cpu().numpy().view(np.uint32)


# ---------------------------------------------------------------------------- bit-identical to the batch ----
@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPH_NAMES)
def test_rows_are_the_dense_batch_top(sp, cuda, name):
    import torch
    n, (rp, ci, va) = _graphs()[name]
    G = _device_graph(sp, cuda, n, rp, ci, va)
    pool = _columns(n, rp, ci, va, 20, seed=len(name) + 3)
    cfg = sp.make_pagerank_config(D, 1e-7, 300)
    tops = sorted({t for t in (1, 10, 100, n, n + 3) if t <= 1024} | ({1024} if n + 3 > 1024 else set()))
    for k in (1, 8, 9, 20):
        V = pool[:k]
        ranks, it, res, conv, hist = sp.pagerank_personalized_batch(G.ptr, V, cfg, capacity=40)
        dense = ranks.cpu().numpy()
        for top in tops:
            ids, vals, it2, res2, conv2, hist2 = sp.pagerank_personalized_batch_top_k(G.ptr, V, top, cfg, capacity=40)
            assert ids.shape == (k, top) and vals.shape == (k, top) and ids.dtype == torch.int32
            assert np.array_equal(it2, it) and np.array_equal(res2.view(np.uint32), res.view(np.uint32))
            assert np.array_equal(conv2, conv) and np.array_equal(hist2, hist, equal_nan=True)
            h_ids, h_vals = ids.cpu().numpy(), vals.cpu().numpy()
            for c in range(k):
                what = f"{name} k={k} top={top} row {c}"
                _assert_row(h_ids[c], h_vals[c], dense[:, c], top, what)
                d_ids, d_vals = sp.pagerank_top_k_device(ranks[:, c].contiguous(), top)
                kk = min(top, n)
                assert np.array_equal(h_ids[c, :kk], d_ids) and np.array_equal(h_vals[c, :kk].view(np.uint32),
                                                                              d_vals.view(np.uint32)), what
                assert (h_ids[c, kk:] == -1).all() and (h_vals[c, kk:].view(np.uint32) == 0).all(), what


@pytest.mark.gpu
def test_api_forms_and_non_square(sp, cuda):
    """Seed ids, dense and scipy.sparse V give the same rows; a non-square adjacency is INVALID_DIMENSION with the
    results zeroed and the output arrays untouched."""
    import scipy.sparse as S
    import torch
    n, rp, ci, va = rmat(11, 8, 72)
    G = _device_graph(sp, cuda, n, rp, ci, va)
    seeds = np.array([0, 5, n - 1, 17, 300, 1000, 2, 9, 44], np.int64)
    dense = np.zeros((seeds.size, n), np.float32)
    dense[np.arange(seeds.size), seeds] = 1.0
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    ref = sp.pagerank_personalized_batch_top_k(G.ptr, seeds, 37, cfg)
    for V in (dense, S.csr_matrix(dense)):
        got = sp.pagerank_personalized_batch_top_k(G.ptr, V, 37, cfg)
        assert torch.equal(got[0], ref[0]) and np.array_equal(_bits(got[1]), _bits(ref[1])) and np.array_equal(got[2], ref[2])
    R = sp.DeviceCSR(n, n + 1, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    d_ids = torch.full((2, 5), 7, dtype=torch.int32, device=cuda)
    d_vals = torch.full((2, 5), 7.0, device=cuda)
    rc, it, res, conv, _ = _call(sp, R.ptr, 2, [0, 1, 2], [0, 1], None, cfg, 5, sp.dptr(d_ids), sp.dptr(d_vals))
    assert rc == int(sp.SpMVError.INVALID_DIMENSION) and (it == 0).all() and (res == 0).all() and not conv.any()
    assert (d_ids == 7).all() and (d_vals == 7.0).all()


# ----------------------------------------------------------------------------------------------- ties ----
@pytest.mark.gpu
def test_ties_fill_in_ascending_node_order(sp, cuda):
    # max_iterations = 0: every rank is the same, so each row is nodes 0 .. top-1
    n, (rp, ci, va) = _graphs()["rmat10"]
    G = _device_graph(sp, cuda, n, rp, ci, va)
    seeds = np.array([3, 900, 17, 4, 5, 6, 7, 8, 1000], np.int64)
    cfg = sp.make_pagerank_config(D, 1e-6, 0)
    ranks = sp.pagerank_personalized_batch(G.ptr, seeds, cfg)[0].cpu().numpy()
    ids, vals = (t.cpu().numpy() for t in sp.pagerank_personalized_batch_top_k(G.ptr, seeds, 100, cfg)[:2])
    assert (ids == np.arange(100, dtype=np.int32)).all()
    assert np.array_equal(vals.view(np.uint32), np.broadcast_to(ranks[:100].T, vals.shape).view(np.uint32))

    # a directed cycle with a uniform teleport vector: every rank is equal at every iteration
    m = 50
    rp, ci, va = graph(m, [(i, (i + 1) % m) for i in range(m)])
    C_ = _device_graph(sp, cuda, m, rp, ci, va)
    V = np.ones((3, m), np.float32)
    cfg = sp.make_pagerank_config(D, 0.0, 20)
    ranks = sp.pagerank_personalized_batch(C_.ptr, V, cfg)[0].cpu().numpy()
    assert (ranks == ranks[0, 0]).all()
    for top in (1, 10, m, m + 3):
        ids, vals = (t.cpu().numpy() for t in sp.pagerank_personalized_batch_top_k(C_.ptr, V, top, cfg)[:2])
        for c in range(3):
            _assert_row(ids[c], vals[c], ranks[:, c], top, f"cycle top={top} row {c}")

    # two copies of a tree in which every node has one in-edge: node j and node j + h rank the same bit for bit
    # (a one-entry row sum has no order), so the K-th and (K+1)-th ranks are equal for some odd K
    rng = np.random.default_rng(5)
    h = 300
    parent = [int(rng.integers(0, j)) for j in range(1, h)]
    edges = [(p, j) for j, p in zip(range(1, h), parent)]
    edges += [(p + h, j + h) for p, j in edges]
    rp, ci, va = graph(2 * h, edges)
    T = _device_graph(sp, cuda, 2 * h, rp, ci, va)
    w = rng.uniform(0.5, 2.0, h).astype(np.float32)
    V = np.stack([np.ones(2 * h, np.float32), np.concatenate([w, w])])
    cfg = sp.make_pagerank_config(D, 1e-7, 200)
    ranks = sp.pagerank_personalized_batch(T.ptr, V, cfg)[0].cpu().numpy()
    assert np.array_equal(ranks[:h].view(np.uint32), ranks[h:].view(np.uint32))
    for c in range(2):
        srt = np.sort(ranks[:, c])[::-1]
        straddle = [t for t in range(1, 200) if srt[t - 1] == srt[t]]
        assert straddle, c
        for top in straddle[:4] + [101]:
            ids, vals = (t.cpu().numpy() for t in sp.pagerank_personalized_batch_top_k(T.ptr, V, top, cfg)[:2])
            _assert_row(ids[c], vals[c], ranks[:, c], top, f"tree top={top} row {c}")


# ------------------------------------------------------------------------- independence, determinism ----
@pytest.mark.gpu
def test_a_row_does_not_depend_on_the_batch(sp, cuda):
    n, (rp, ci, va) = _graphs()["rmat12"]
    G = _device_graph(sp, cuda, n, rp, ci, va)
    pool = _columns(n, rp, ci, va, 20, seed=5)
    cfg = sp.make_pagerank_config(D, 1e-6, 200)

    def run(V):
        ids, vals, it, res, conv, hist = sp.pagerank_personalized_batch_top_k(G.ptr, V, 64, cfg, capacity=200)
        return ids.cpu().numpy(), _bits(vals), it, res, conv, hist

    full_a, full_b = run(pool), run(pool)
    for x, y in zip(full_a, full_b):  # two runs
        assert np.array_equal(x, y, equal_nan=True) if x.dtype.kind == "f" else np.array_equal(x, y)
    perm = [19, 3, 17, 0, 11, 6, 16, 9]  # rows from every chunk of the k = 20 run, at other positions
    mixed = run(pool[perm])
    for pos, c in enumerate(perm):
        alone = run(pool[c:c + 1])
        for got, j in ((mixed, pos), (full_a, c)):
            for x, y in zip(got, alone):
                assert np.array_equal(x[j], y[0], equal_nan=True) if x.dtype.kind == "f" else np.array_equal(x[j], y[0]), (c, j)


# ------------------------------------------------------------------------------------ past the memory wall ----
@pytest.mark.gpu
def test_more_seeds_than_a_dense_output_could_hold(sp, cuda):
    """k one-hot seeds on R-MAT 20 with n * k * 4 bytes above the device's memory: the call runs, and its first,
    middle and last rows are those of the dense batch run on those three seeds alone."""
    import torch
    n, rp, ci, va = rmat(20, 4, 73)
    G = _device_graph(sp, cuda, n, rp, ci, va)
    total = torch.cuda.mem_get_info()[1]
    k = math.ceil(1.05 * total / (4 * n))
    assert k * n * 4 > total and k <= n
    seeds = (np.arange(k, dtype=np.int64) * 7919) % n  # distinct: 7919 is odd, n a power of two
    cfg = sp.make_pagerank_config(D, 0.0, 2)
    ids, vals, it, res, conv, _ = sp.pagerank_personalized_batch_top_k(G.ptr, seeds, 8, cfg)
    assert (it == 2).all() and not conv.any()
    pick = [0, k // 2, k - 1]
    ranks, it3, res3 = sp.pagerank_personalized_batch(G.ptr, seeds[pick], cfg)[:3]
    dense = ranks.cpu().numpy()
    for j, c in enumerate(pick):
        _assert_row(ids[c].cpu().numpy(), vals[c].cpu().numpy(), dense[:, j], 8, f"seed row {c} of {k}")
        assert res[c] == res3[j]


# ---------------------------------------------------------------------------------------------- kernels ----
@pytest.mark.gpu
def test_call_launches_every_library_kernel(sp, cuda):
    """Under torch.profiler, the kernels of a top-K call (k = 9: two chunks) that are not libspmv_b200.so's are exactly
    the kernels libspmv_b200_ppr_topk.so ships, and those are none of libspmv_b200.so's."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    n, rp, ci, va = rmat(13, 8, 71)
    G = _device_graph(sp, cuda, n, rp, ci, va)
    V = _columns(n, rp, ci, va, 9, seed=9)
    before = sp.ppr_topk_lib().spmv_b200_ppr_topk_launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sp.pagerank_personalized_batch_top_k(G.ptr, V, 10, sp.make_pagerank_config(D, 1e-6, 100))
        torch.cuda.synchronize()
    assert sp.ppr_topk_lib().spmv_b200_ppr_topk_launch_count() > before
    ss = _sass_summary()
    shipped = ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200_ppr_topk.so"))
    main = ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200.so"))
    assert shipped and not (shipped & main)
    assert "ppr::ppr_scale_kernel" not in shipped
    names = sorted({ev.name for ev in prof.events() if ev.device_type == DeviceType.CUDA})
    if not names:
        pytest.skip("the profiler records no CUDA kernels on this machine")
    launched = {k for k in ss.demangle(names) if not k.startswith(("Memcpy", "Memset"))}
    assert launched - main == shipped, f"launched {sorted(launched - main)}, shipped {sorted(shipped)}"


def test_importing_the_package_does_not_load_the_library():
    code = ("import _load_pkg; _load_pkg.load_pkg(); "
            "print(any('libspmv_b200_ppr_topk' in line for line in open('/proc/self/maps')))")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, check=True)
    assert out.stdout.strip() == "False"
