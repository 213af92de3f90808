"""Batched personalized PageRank (libspmv_b200_ppr.so): k teleport vectors per pass over the graph.

- Every column c is within L1 1e-6 of orc_pagerank_personalized_f64 at c's own iteration count, its converged ranks
  are the exact fixed point to within the error the stop rule allows, and its iteration count is within 1 of the
  oracle's own stop.
- A column's result does not depend on the batch: alone, at another position of a chunk, in a later chunk and in a
  second run it is the same bit for bit, and a column that converges early keeps its vector while the others iterate.
- API behaviour: max_iterations = 0, an unreachable tolerance, per-column residual history, n = 0, a non-square
  adjacency.
- The companion ships exactly the kernels a batch launches, and exports exactly the functions of its header.
- Input validation needs no GPU and launches nothing."""
import ctypes as C
import functools
import os
import re
import subprocess

import numpy as np
import pytest

from test_gpu_pagerank_personalized import _sass_summary, dangling, exact_fixed_point, graph, orc_personalized, rmat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "gpu-spmv_b200", "lib")
D = 0.85


def _call(sp, A, k, offsets, nodes, weights, cfg, d_ranks=None, capacity=0):
    """The C entry point with raw arrays -> (rc, iterations, residual, converged, history)."""
    ip, fp = C.POINTER(C.c_int), C.POINTER(C.c_float)
    kk = max(k, 1)
    it, res, conv = np.zeros(kk, np.int32), np.zeros(kk, np.float32), np.zeros(kk, np.bool_)
    hist = np.full(kk * max(capacity, 1), np.nan, np.float32)
    arr = lambda a, t, p: np.ascontiguousarray(a, t).ctypes.data_as(p) if a is not None else None  # noqa: E731
    rc = sp.ppr_lib().spmv_b200_pagerank_personalized_batch(
        A, C.byref(cfg) if cfg is not None else None, k, arr(offsets, np.int32, ip), arr(nodes, np.int32, ip),
        arr(weights, np.float32, fp), d_ranks, it.ctypes.data_as(ip), res.ctypes.data_as(fp),
        conv.ctypes.data_as(C.POINTER(C.c_bool)), hist.ctypes.data_as(fp) if capacity > 0 else None, capacity)
    return rc, it, res, conv, hist


# -------------------------------------------------------------------------------- input validation (CPU) ----
def test_rejected_inputs_launch_nothing(sp):
    """Every malformed batch is INVALID_ARGUMENT before any device work.  The CSR has host arrays only and d_ranks
    is a bogus non-NULL address: nothing could run anyway, and neither library's launch counter moves."""
    bad_arg = int(sp.SpMVError.INVALID_ARGUMENT)
    n = 4
    A = sp.csr_create(0, 0, 0)
    sp.csr_from_dense(A, np.eye(n, dtype=np.float32), n, n)
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    fake = C.c_void_p(0x1000)
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
    before, before_ppr = sp.launch_count(), sp.ppr_lib().spmv_b200_ppr_launch_count()
    for name, (k, off, nodes, w) in cases.items():
        assert _call(sp, A, k, off, nodes, w, cfg, fake)[0] == bad_arg, name
    good = ([0, 1, 3], [2, 0, 3], [1.0, 2.0, 0.5])
    assert _call(sp, None, 2, *good, cfg, fake)[0] == bad_arg  # NULL adjacency
    assert _call(sp, A, 2, *good, cfg, None)[0] == bad_arg  # NULL d_ranks
    assert _call(sp, None, 2, None, None, None, cfg, fake)[0] == bad_arg  # NULL offsets
    f = sp.ppr_lib().spmv_b200_pagerank_personalized_batch
    off, nod = np.array(good[0], np.int32), np.array(good[1], np.int32)
    ip = C.POINTER(C.c_int)
    it, res, conv = np.zeros(2, np.int32), np.zeros(2, np.float32), np.zeros(2, np.bool_)
    args = [off.ctypes.data_as(ip), nod.ctypes.data_as(ip), None, fake]
    outs = [it.ctypes.data_as(ip), res.ctypes.data_as(C.POINTER(C.c_float)), conv.ctypes.data_as(C.POINTER(C.c_bool))]
    for i in range(3):  # each NULL result array
        o = list(outs)
        o[i] = None
        assert f(A, C.byref(cfg), 2, *args, *o, None, 0) == bad_arg, i
    assert f(A, C.byref(cfg), 2, *args, *outs, None, 4) == bad_arg  # history capacity without a history array
    assert f(A, C.byref(cfg), 2, *args, *outs, None, -1) == bad_arg
    # n = 0: every column is necessarily empty (the single-vector call rejects an n = 0 vector the same way)
    Z = sp.csr_create(0, 0, 0)
    assert _call(sp, Z, 1, [0, 0], [], None, cfg, fake)[0] == bad_arg
    assert _call(sp, Z, 1, [0, 1], [0], None, cfg, fake)[0] == bad_arg
    with pytest.raises(RuntimeError):
        sp.pagerank_personalized_batch(A, np.array([[1.0, np.nan, 0, 0]], np.float32), cfg)
    with pytest.raises(ValueError):
        sp.pagerank_personalized_batch(A, np.ones((2, n + 1), np.float32), cfg)  # the shape is checked in Python
    assert sp.launch_count() == before
    assert sp.ppr_lib().spmv_b200_ppr_launch_count() == before_ppr
    sp.csr_destroy(A)
    sp.csr_destroy(Z)


def test_companion_exports_exactly_its_header(sp):
    sp.ppr_lib()  # built and loadable
    header = open(os.path.join(ROOT, "include", "spmv_b200_ppr.h")).read()
    declared = set(re.findall(r"SPMV_B200_API[^;(]*?\b(spmv_b200_\w+)\s*\(", header))
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(LIBDIR, "libspmv_b200_ppr.so")],
                         capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if line.split() and line.split()[-2] in "TtWwDdBbRrVvi"}
    assert declared == {"spmv_b200_pagerank_personalized_batch", "spmv_b200_ppr_launch_count"}
    assert exported == declared


# --------------------------------------------------------------------------------------------- helpers ----
@functools.lru_cache(maxsize=None)
def _graphs():
    g = {}
    g["dense4"] = (4, graph(4, [(0, 1), (1, 2), (2, 0), (2, 3), (3, 0), (0, 2)]))
    g["dense5_dangling"] = (5, graph(5, [(0, 1), (1, 2), (2, 0), (3, 4), (0, 4), (2, 3)]))
    g["dense6"] = (6, graph(6, [(a, b) for a in range(6) for b in range(6) if a != b and (a * 7 + b * 3) % 4 != 0]))
    g["dangling_isolated8"] = (8, graph(8, [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 4), (1, 6), (4, 6), (2, 5)]))
    for scale, seed in ((8, 61), (10, 62), (12, 63), (14, 64)):
        n, rp, ci, va = rmat(scale, 8, seed)
        g[f"rmat{scale}"] = (n, (rp, ci, va))
    return g


GRAPH_NAMES = ["dense4", "dense5_dangling", "dense6", "dangling_isolated8", "rmat8", "rmat10", "rmat12", "rmat14"]


def _columns(n, rp, ci, va, count=20, seed=0):
    """`count` dense teleport vectors: single seeds, seed sets, a dangling seed, uniform, mixed weights."""
    rng = np.random.default_rng(seed)
    delta = dangling(n, rp, ci, va)
    cols = []
    for j in range(count):
        v = np.zeros(n, np.float32)
        kind = j % 5
        if kind == 0:
            v[(j * 7919) % n] = 1.0
        elif kind == 1:
            idx = rng.choice(n, min(n, 3 + j % 4), replace=False)
            v[idx] = rng.uniform(0.5, 2.0, idx.size)
        elif kind == 2:
            v[np.flatnonzero(delta)[j % max(1, delta.sum())] if delta.any() else n - 1] = 2.0
        elif kind == 3:
            v[:] = 1.0
        else:
            v[:] = rng.uniform(0.0, 1.0, n) * (rng.random(n) < 0.2)
            v[rng.integers(0, n)] = 0.75
        cols.append(v)
    return np.stack(cols)


def _device_graph(sp, cuda, n, rp, ci, va):
    import torch
    return sp.DeviceCSR(n, n, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))


# ---------------------------------------------------------------------------------------------- oracle ----
@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPH_NAMES)
def test_every_column_matches_the_oracle(sp, cuda, name):
    n, (rp, ci, va) = _graphs()[name]
    G = _device_graph(sp, cuda, n, rp, ci, va)
    pool = _columns(n, rp, ci, va, 20, seed=len(name))
    tol, cap = 1e-7, 500
    cfg = sp.make_pagerank_config(D, tol, cap)
    differ = 0
    for k in (1, 3, 8, 9, 20):
        V = pool[:k]
        ranks, iters, res, conv, _ = sp.pagerank_personalized_batch(G.ptr, V, cfg)
        ranks = ranks.cpu().numpy().astype(np.float64)
        for c in range(k):
            assert iters[c] > 0, (name, k, c)
            o_at, _, _, o_l1, _ = orc_personalized(n, rp, ci, va, V[c], tol=tol, max_it=cap, fixed_it=int(iters[c]))
            err = float(np.abs(ranks[:, c] - o_at).sum())
            assert err <= 1e-6, f"{name} k={k} column {c}: L1 {err:.3e} to the restatement after {iters[c]} iterations"
            o_it, o_conv = orc_personalized(n, rp, ci, va, V[c], tol=tol, max_it=cap)[1::3]
            assert abs(int(iters[c]) - o_it) <= 1 and bool(conv[c]) == o_conv, (name, k, c, iters[c], o_it)
            differ += int(iters[c]) != o_it
            if n <= 4096:
                exact = exact_fixed_point(n, rp, ci, va, V[c])
                bound = D / (1 - D) * o_l1 + 2e-6
                err = float(np.abs(ranks[:, c] - exact).sum())
                assert err <= bound, f"{name} k={k} column {c}: L1 {err:.3e} to the fixed point, bound {bound:.3e}"
    print(f"{name}: {differ} of {1 + 3 + 8 + 9 + 20} columns stopped one iteration away from the oracle")


# ------------------------------------------------------------------------- independence, determinism ----
@pytest.mark.gpu
def test_a_column_does_not_depend_on_the_batch(sp, cuda):
    n, (rp, ci, va) = _graphs()["rmat12"]
    G = _device_graph(sp, cuda, n, rp, ci, va)
    pool = _columns(n, rp, ci, va, 20, seed=5)
    cfg = sp.make_pagerank_config(D, 1e-6, 200)

    def run(V):
        r, it, res, conv, hist = sp.pagerank_personalized_batch(G.ptr, V, cfg, capacity=200)
        return r.cpu().numpy().view(np.uint32), it, res, conv, hist

    full_a, full_b = run(pool), run(pool)
    for x, y in zip(full_a, full_b):  # two runs
        assert np.array_equal(x, y, equal_nan=True) if x.dtype.kind == "f" else np.array_equal(x, y)
    perm = [19, 3, 17, 0, 11, 6, 16, 9]  # columns from every chunk of the k = 20 run, at other positions
    mixed = run(pool[perm])
    for pos, c in enumerate(perm):
        alone = run(pool[c:c + 1])
        for got, lbl in ((mixed, f"position {pos} of k = 8"), (full_a, f"column {c} of k = 20")):
            j = pos if got is mixed else c
            assert np.array_equal(got[0][:, j], alone[0][:, 0]), f"column {c} ranks: {lbl} differs from alone"
            assert got[1][j] == alone[1][0] and got[2][j] == alone[2][0] and got[3][j] == alone[3][0], (c, lbl)
            assert np.array_equal(got[4][j], alone[4][0], equal_nan=True), (c, lbl)
    # a column that converged early kept its vector while the others of its chunk iterated on
    it = full_a[1]
    early = [c for c in range(20) if it[c] < it[(c // 8) * 8:(c // 8) * 8 + 8].max()]
    assert early, it
    assert it.min() < it.max()


# ------------------------------------------------------------------------------------------------- API ----
@pytest.mark.gpu
def test_api_edges(sp, cuda):
    import torch
    scale = 11
    n, rp, ci, va = rmat(scale, 8, 70)
    G = _device_graph(sp, cuda, n, rp, ci, va)
    seeds = np.array([0, 5, n - 1, 17, 300, 1000, 2, 9, 44], np.int64)
    # max_iterations = 0: the uniform start vector, normalised
    ranks, it, res, conv, _ = sp.pagerank_personalized_batch(G.ptr, seeds, sp.make_pagerank_config(D, 1e-6, 0))
    assert (it == 0).all() and (res == 0).all() and not conv.any()
    assert np.array_equal(ranks.cpu().numpy(), np.full((n, seeds.size), 1.0 / n, np.float32))
    # an unreachable tolerance runs every column to the cap
    ranks, it, res, conv, hist = sp.pagerank_personalized_batch(G.ptr, seeds, sp.make_pagerank_config(D, 0.0, 25), capacity=30)
    assert (it == 25).all() and not conv.any() and np.isfinite(hist[:, :25]).all() and np.isnan(hist[:, 25:]).all()
    for c, s in enumerate(seeds):  # one-hot columns = the single-vector call with the same vector
        v = np.zeros(n, np.float32)
        v[s] = 1.0
        o = orc_personalized(n, rp, ci, va, v, tol=0.0, max_it=25, fixed_it=25)[0]
        assert float(np.abs(ranks[:, c].cpu().numpy().astype(np.float64) - o).sum()) <= 1e-6
        assert hist[c, 24] == res[c]
    # each column's history ends at its first value below the tolerance
    tol = 1e-6
    ranks, it, res, conv, hist = sp.pagerank_personalized_batch(G.ptr, seeds, sp.make_pagerank_config(D, tol, 100), capacity=100)
    assert conv.all()
    for c in range(seeds.size):
        h = hist[c]
        assert (h[:it[c] - 1] >= np.float32(tol)).all() and h[it[c] - 1] < np.float32(tol) and h[it[c] - 1] == res[c]
        assert np.isnan(h[it[c]:]).all()
    # the same vectors given densely and as scipy.sparse give the same bits
    import scipy.sparse as S
    dense = np.zeros((seeds.size, n), np.float32)
    dense[np.arange(seeds.size), seeds] = 1.0
    for V in (dense, S.csr_matrix(dense)):
        r2, it2 = sp.pagerank_personalized_batch(G.ptr, V, sp.make_pagerank_config(D, tol, 100))[:2]
        assert np.array_equal(it2, it) and np.array_equal(r2.cpu().numpy().view(np.uint32), ranks.cpu().numpy().view(np.uint32))
    # non-square adjacency: INVALID_DIMENSION, as the single-vector call; results zeroed
    R = sp.DeviceCSR(n, n + 1, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    d = torch.full((n, 2), 7.0, device=cuda)
    rc, it, res, conv, _ = _call(sp, R.ptr, 2, [0, 1, 2], [0, 1], None, sp.make_pagerank_config(D, 1e-6, 100), sp.dptr(d))
    assert rc == int(sp.SpMVError.INVALID_DIMENSION) and (it == 0).all() and not conv.any()
    assert (d == 7.0).all()
    v = np.zeros(n, np.float32)
    v[0] = 1.0
    assert sp.pagerank_device_personalized(R.ptr, torch.empty(n, device=cuda), v)[0] == int(sp.SpMVError.INVALID_DIMENSION)


# ---------------------------------------------------------------------------------- companion kernels ----
@pytest.mark.gpu
def test_batch_launches_every_companion_kernel(sp, cuda):
    """Under torch.profiler, the kernels of a batch (k = 9: two chunks, columns converging at different
    iterations) that are not libspmv_b200.so's are exactly the kernels libspmv_b200_ppr.so ships."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    n, rp, ci, va = rmat(13, 8, 71)
    G = _device_graph(sp, cuda, n, rp, ci, va)
    V = _columns(n, rp, ci, va, 9, seed=9)
    before = sp.ppr_lib().spmv_b200_ppr_launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ranks, it = sp.pagerank_personalized_batch(G.ptr, V, sp.make_pagerank_config(D, 1e-6, 100))[:2]
        torch.cuda.synchronize()
    assert sp.ppr_lib().spmv_b200_ppr_launch_count() > before
    assert it.min() < it.max()
    ss = _sass_summary()
    shipped = ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200_ppr.so"))
    main = ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200.so"))
    assert shipped and not (shipped & main)
    names = sorted({ev.name for ev in prof.events() if ev.device_type == DeviceType.CUDA})
    if not names:
        pytest.skip("the profiler records no CUDA kernels on this machine")
    launched = {k for k in ss.demangle(names) if not k.startswith(("Memcpy", "Memset"))}
    assert launched - main == shipped, f"launched {sorted(launched - main)}, shipped {sorted(shipped)}"
