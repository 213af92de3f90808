"""Personalized PageRank: teleport and dangling mass follow a caller-given vector v (normalised to v / sum(v)).

- The converged ranks are the exact fixed point: the solution of (I - d A - d v delta^T) r = (1 - d) v with
  sum(r) = 1 (delta = dangling indicator), solved in f64 with scipy, to within the error the stop rule allows.
- Every kernel path (one-kernel loop, plain tile, hub plan, segmented stream, sharded with 2 and 3 ranks on one
  GPU) is within L1 1e-6 of orc_pagerank_personalized_f64 (tests/pagerank_personalized_oracle.c, the f64-accumulator
  restatement in the style of oracle/spmv_oracle.c) at the same iteration count, and
  launches the same kernels as its uniform twin.  The tuning variables are read once per process, so every path
  runs in a child process (this file with --child), as in test_gpu_kernel_coverage.py.
- API behaviour: stop rule, max_iterations = 0, residual history, device top-k, the drop-in host call.
- The sharded object: setting and clearing v gives back the global vector bit for bit (the cached iteration
  graphs are captured again).
- Input validation needs no GPU and launches nothing."""
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
D = 0.85


# ------------------------------------------------------------------------------------------------ helpers ----
@functools.lru_cache(maxsize=None)
def _personalized_oracle():
    """tests/pagerank_personalized_oracle.c, compiled into a temporary directory (the tree may be read-only) with
    the flags of oracle/Makefile."""
    import tempfile
    out = os.path.join(tempfile.mkdtemp(prefix="ppr_oracle_"), "libppr_oracle.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fvisibility=hidden", "-shared",
                           "-fPIC", "-o", out, os.path.join(ROOT, "tests", "pagerank_personalized_oracle.c"), "-lm"])
    return C.CDLL(out)


def orc_personalized(n, rp, ci, va, v, damping=D, tol=1e-6, max_it=100, fixed_it=0):
    """orc_pagerank_personalized_f64 -> (ranks, iterations, l2, l1, converged)."""
    fp, ip, dp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)
    f = _personalized_oracle().orc_pagerank_personalized_f64
    f.argtypes = [C.c_int, C.c_int, fp, ip, ip, fp, C.c_float, C.c_float, C.c_int, C.c_int, fp, dp, dp, ip]
    rp, ci = np.ascontiguousarray(rp, np.int32), np.ascontiguousarray(ci, np.int32)
    va, v = np.ascontiguousarray(va, np.float32), np.ascontiguousarray(v, np.float32)
    ranks = np.empty(n, np.float32)
    l2, l1, conv = C.c_double(0), C.c_double(0), C.c_int(0)
    it = f(n, n, va.ctypes.data_as(fp), ci.ctypes.data_as(ip), rp.ctypes.data_as(ip), v.ctypes.data_as(fp), damping, tol,
           max_it, fixed_it, ranks.ctypes.data_as(fp), C.byref(l2), C.byref(l1), C.byref(conv))
    assert it >= 0, "the oracle rejected the personalization vector"
    return ranks, it, l2.value, l1.value, bool(conv.value)


def graph(n, edges):
    """Column-normalised adjacency of a directed graph (row = dst, col = src, value 1/outdeg(src)), as pagerank()
    expects.  Returns (rp, ci, va)."""
    src = np.array([e[0] for e in edges], np.int64)
    dst = np.array([e[1] for e in edges], np.int64)
    outdeg = np.bincount(src, minlength=n)
    order = np.lexsort((src, dst))
    src, dst = src[order], dst[order]
    rp = np.zeros(n + 1, np.int32)
    rp[1:] = np.cumsum(np.bincount(dst, minlength=n))
    return rp, src.astype(np.int32), (1.0 / outdeg[src]).astype(np.float32)


def rmat(scale, ef, seed):
    import gpu_spmv_b200.gen as gen
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, ef, seed, "cpu")
    return n, rp.numpy(), ci.numpy(), va.numpy()


def dangling(n, rp, ci, va):
    colsum = np.zeros(n)
    np.add.at(colsum, ci, va.astype(np.float64))
    return colsum == 0


def random_personalization(n, seed):
    """Non-negative, mostly zero, at least one positive entry."""
    rng = np.random.default_rng(seed)
    v = (rng.uniform(0.0, 3.0, n) * (rng.random(n) < 0.3)).astype(np.float32)
    v[rng.integers(0, n)] = 1.0
    return v


def exact_fixed_point(n, rp, ci, va, v, damping=D):
    """Solution of (I - d A - d vhat delta^T) r = (1 - d) vhat, scaled to sum(r) = 1, in f64.

    With B = I - d A and x = B^-1 vhat, Sherman-Morrison gives r = (1 - d) x / (1 - d delta^T x): one sparse solve,
    no dense outer product.  The stated system is checked on the result."""
    import scipy.sparse as S
    import scipy.sparse.linalg as SL
    A = S.csr_matrix((va.astype(np.float64), ci, rp), shape=(n, n))
    vhat = v.astype(np.float64) / v.astype(np.float64).sum()
    delta = dangling(n, rp, ci, va)
    x = SL.spsolve((S.identity(n, format="csc") - damping * A).tocsc(), vhat)
    r = (1 - damping) * x / (1 - damping * x[delta].sum())
    lhs = r - damping * (A @ r) - damping * vhat * r[delta].sum()
    assert np.abs(lhs - (1 - damping) * vhat).max() <= 1e-12
    return r / r.sum()


def _sass_summary():
    spec = importlib.util.spec_from_file_location("sass_summary", os.path.join(ROOT, "scripts", "sass_summary.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# -------------------------------------------------------------------------------- input validation (CPU) ----
def test_rejected_personalization_vectors_launch_nothing(sp):
    """NaN, +-Inf, a negative entry and an all-zero vector are INVALID_ARGUMENT before any device work, and so are
    a NULL adjacency and a NULL sharded handle.  The CSR here has host arrays only: nothing could run anyway."""
    bad_arg = int(sp.SpMVError.INVALID_ARGUMENT)
    n = 4
    A = sp.csr_create(0, 0, 0)
    sp.csr_from_dense(A, np.eye(n, dtype=np.float32), n, n)
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    res = sp.PageRankResult()
    ranks = np.empty(n, np.float32)
    import gpu_spmv_b200.dist as Dm
    dres = Dm.PrDistResult()
    fp = C.POINTER(C.c_float)
    good = np.array([1, 0, 2, 0], np.float32)
    bad = {"nan": [1, np.nan, 1, 1], "+inf": [1, np.inf, 0, 0], "-inf": [0, 0, -np.inf, 1], "negative": [1, 2, -1e-30, 1],
           "zero": [0, 0, 0, 0], "negative zero only": [-0.0, 0, 0, 0]}
    before = sp.launch_count()
    for name, v in bad.items():
        v = np.array(v, np.float32)
        p = v.ctypes.data_as(fp)
        assert sp.lib.spmv_b200_pagerank_personalized(A, C.byref(cfg), p, C.byref(res)) == bad_arg, name
        assert not res.ranks, name
        assert sp.lib.spmv_b200_pagerank_device_personalized(A, C.byref(cfg), p, 16, None, None, None, None, None,
                                                             0) == bad_arg, name
        assert sp.lib.spmv_b200_pagerank_multi_personalized(A, C.byref(cfg), p, 2, None, 1, 4, 0,
                                                            ranks.ctypes.data_as(C.c_void_p), C.byref(dres)) == bad_arg, name
        with pytest.raises(RuntimeError):
            sp.pagerank_personalized(A, v, cfg)
    gp = good.ctypes.data_as(fp)
    assert sp.lib.spmv_b200_pagerank_personalized(None, C.byref(cfg), gp, C.byref(res)) == bad_arg
    assert sp.lib.spmv_b200_pagerank_device_personalized(None, C.byref(cfg), gp, 16, None, None, None, None, None, 0) == bad_arg
    assert sp.lib.spmv_b200_pagerank_multi_personalized(None, C.byref(cfg), gp, 2, None, 1, 4, 0,
                                                        ranks.ctypes.data_as(C.c_void_p), C.byref(dres)) == bad_arg
    assert sp.lib.spmv_b200_pr_dist_set_personalization(None, gp) == bad_arg
    assert sp.lib.spmv_b200_pr_dist_set_personalization(None, None) == bad_arg
    with pytest.raises(ValueError):
        sp.pagerank_personalized(A, np.ones(n + 1, np.float32), cfg)  # the length is checked in Python
    assert sp.launch_count() == before
    sp.csr_destroy(A)


# ------------------------------------------------------------------------------------------- fixed point ----
@functools.lru_cache(maxsize=None)
def _small_graphs():
    g = {}
    g["dense4"] = (4, graph(4, [(0, 1), (1, 2), (2, 0), (2, 3), (3, 0), (0, 2)]))
    g["dense5_dangling"] = (5, graph(5, [(0, 1), (1, 2), (2, 0), (3, 4), (0, 4), (2, 3)]))  # 4 has no out-links
    g["dense6"] = (6, graph(6, [(a, b) for a in range(6) for b in range(6) if a != b and (a * 7 + b * 3) % 4 != 0]))
    # 6 is dangling (in-links, no out-links), 7 is isolated (neither)
    g["dangling_isolated8"] = (8, graph(8, [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 4), (1, 6), (4, 6), (2, 5)]))
    for scale, seed in ((8, 21), (10, 22), (12, 23)):
        n, rp, ci, va = rmat(scale, 8, seed)
        g[f"rmat{scale}"] = (n, (rp, ci, va))
    return g


def _personalizations(n, rp, ci, va):
    delta = dangling(n, rp, ci, va)
    seed_set = np.zeros(n, np.float32)
    seed_set[[0, n // 2, n - 1]] = [1.0, 2.0, 0.5]
    single = np.zeros(n, np.float32)
    single[1] = 3.0
    dseed = np.zeros(n, np.float32)
    dseed[np.flatnonzero(delta)[0] if delta.any() else n - 1] = 1.0
    return {"single_seed": single, "seed_set": seed_set, "dangling_seed": dseed, "uniform": np.ones(n, np.float32)}


GRAPH_NAMES = ["dense4", "dense5_dangling", "dense6", "dangling_isolated8", "rmat8", "rmat10", "rmat12"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPH_NAMES)
def test_converged_ranks_are_the_exact_fixed_point(sp, orc, cuda, name):
    import torch
    n, (rp, ci, va) = _small_graphs()[name]
    G = sp.DeviceCSR(n, n, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    d_ranks = torch.empty(n, dtype=torch.float32, device=cuda)
    cfg = sp.make_pagerank_config(D, 1e-7, 500)
    for label, v in _personalizations(n, rp, ci, va).items():
        rc, iters, res, conv, l1, _ = sp.pagerank_device_personalized(G.ptr, d_ranks, v, cfg)
        assert rc == 0 and iters > 0, (label, rc, iters)
        r = d_ranks.cpu().numpy().astype(np.float64)
        exact = exact_fixed_point(n, rp, ci, va, v)
        # contraction by d in L1: |r_k - r*| <= d / (1 - d) |r_k - r_(k-1)|, plus fp32 rounding of the iterates
        bound = D / (1 - D) * l1 + 2e-6
        err = float(np.abs(r - exact).sum())
        assert err <= bound, f"{name} {label}: L1 {err:.3e} to the exact fixed point, bound {bound:.3e} ({iters} it.)"
        if label == "uniform":
            o_ranks = orc.pagerank_f64(n, n, rp, ci, va, D, 1e-7, 500, fixed_it=iters)[0]
            assert float(np.abs(r - o_ranks).sum()) <= 1e-6, f"{name}: uniform v against global PageRank"


# --------------------------------------------------------------------------- every path, in child processes ----
V = "SPMV_B200_"
PATHS = {
    "small": ({}, (10, 8, 31), 1, ["pagerank_small_kernel"]),
    "tile": ({V + "HOT": "0", V + "PR_SMALL": "0"}, (12, 8, 32), 1,
             ["merge_tile_kernel<PageRankRowT<false>, 7>", "merge_fixup_kernel<PageRankRowT<false>>"]),
    "hub_all_x": ({V + "PLAN": "hub", V + "HOT": "1", V + "PR_SMALL": "0"}, (12, 8, 33), 1,
                  ["merge_hot_kernel<PageRankRowT<true>, true, 7>"]),
    "hub_table": ({V + "PLAN": "hub", V + "HOT": "1", V + "PR_SMALL": "0"}, (17, 4, 34), 1,
                  ["merge_hot_kernel<PageRankRowT<true>, false, 7>"]),
    "seg": ({V + "PLAN": "seg", V + "HOT": "1", V + "PR_SMALL": "0"}, (12, 8, 35), 1, ["seg_pagerank_epilogue_kernel"]),
    "sharded2": ({}, (12, 8, 36), 2, []),
    "sharded3": ({}, (12, 8, 37), 3, []),
}


def _child(path):
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    from _load_pkg import load_pkg
    from oracle_binding import Oracle
    sp, orc = load_pkg(), Oracle()
    import gpu_spmv_b200.dist as Dm
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    _, (scale, ef, seed), world, _ = PATHS[path]
    n, rp, ci, va = rmat(scale, ef, seed)
    v = random_personalization(n, seed)
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    out = {"path": path}
    for label, vec in (("uniform", None), ("personalized", v)):
        got = {}

        def run():
            if world == 1:
                G = sp.DeviceCSR(n, n, torch.as_tensor(rp).to(dev), torch.as_tensor(ci).to(dev), torch.as_tensor(va).to(dev))
                d_ranks = torch.empty(n, dtype=torch.float32, device=dev)
                rc, iters = sp.pagerank_device_personalized(G.ptr, d_ranks, vec, cfg)[:2]
                torch.cuda.synchronize()
                got.update(rc=rc, iters=iters, ranks=d_ranks.cpu().numpy())
            else:
                A = sp.csr_from_arrays(n, n, rp, ci, va)
                ranks = np.empty(n, np.float32)
                res = Dm.PrDistResult()
                devices = (C.c_int * world)(*([0] * world))
                p = vec.ctypes.data_as(C.POINTER(C.c_float)) if vec is not None else None
                rc = sp.lib.spmv_b200_pagerank_multi_personalized(A, C.byref(cfg), p, world, devices, Dm.EXCHANGE_P2P, 4, 0,
                                                                  ranks.ctypes.data_as(C.c_void_p), C.byref(res))
                sp.csr_destroy(A)
                got.update(rc=rc, iters=res.iterations, ranks=ranks, exchange=res.exchange)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run()
            torch.cuda.synchronize()
        names = sorted({ev.name for ev in prof.events() if ev.device_type == DeviceType.CUDA})
        kernels = [k for k in _sass_summary().demangle(names) if not k.startswith(("Memcpy", "Memset"))] if names else []
        if vec is None:
            ref = orc.pagerank_f64(n, n, rp, ci, va, D, 1e-6, 100, fixed_it=max(got["iters"], 1))[0]
        else:
            ref = orc_personalized(n, rp, ci, va, vec, fixed_it=max(got["iters"], 1))[0]
        out[label] = {"rc": got["rc"], "iters": got["iters"], "kernels": sorted(set(kernels)),
                      "l1": float(np.abs(got["ranks"].astype(np.float64) - ref).sum()), "exchange": got.get("exchange")}
    print("PATH " + json.dumps(out), flush=True)


def _run_child(path):
    env = {k: v for k, v in os.environ.items() if not k.startswith(V)}
    env.update(PATHS[path][0])
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    recs = [json.loads(line[5:]) for line in p.stdout.splitlines() if line.startswith("PATH ")]
    assert p.returncode == 0 and len(recs) == 1, p.stdout[-4000:]
    return recs[0]


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_every_path_matches_the_restatement(cuda, path):
    rec = _run_child(path)
    uni, per = rec["uniform"], rec["personalized"]
    for label, r in (("uniform", uni), ("personalized", per)):
        assert r["rc"] == 0 and r["iters"] > 0, (label, r)
        assert r["l1"] <= 1e-6, f"{path} {label}: L1 {r['l1']:.3e} to the f64 restatement after {r['iters']} iterations"
    if PATHS[path][2] > 1:
        assert per["exchange"] == 1 and uni["exchange"] == 1  # peer stores
    if not uni["kernels"] and not per["kernels"]:
        return  # the profiler records no CUDA kernels on this machine
    assert per["kernels"] == uni["kernels"], f"{path}: personalized ran {per['kernels']}, uniform {uni['kernels']}"
    for k in PATHS[path][3]:
        assert k in per["kernels"], f"{path}: expected {k}, ran {per['kernels']}"


# --------------------------------------------------------------------------------------------------- API ----
@pytest.mark.gpu
@pytest.mark.parametrize("scale", [10, 14])
def test_api_stop_rule_history_and_top_k(sp, orc, cuda, scale):
    """scale 10 takes the one-kernel loop, 14 the graph-replayed multi-kernel loop."""
    import torch
    n, rp, ci, va = rmat(scale, 8, 40 + scale)
    v = random_personalization(n, scale)
    G = sp.DeviceCSR(n, n, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    d_ranks = torch.empty(n, dtype=torch.float32, device=cuda)
    rc, iters, res, conv, l1, hist = sp.pagerank_device_personalized(G.ptr, d_ranks, v, sp.make_pagerank_config(D, 1e-6, 100),
                                                                     capacity=100)
    assert rc == 0
    o_ranks, o_it, o_l2, o_l1, o_conv = orc_personalized(n, rp, ci, va, v)
    assert abs(iters - o_it) <= 1 and conv == o_conv, (iters, o_it, conv, o_conv)
    assert np.isfinite(hist[:iters]).all() and np.isnan(hist[iters:]).all()
    assert hist[iters - 1] == np.float32(res)
    o_at = orc_personalized(n, rp, ci, va, v, fixed_it=iters)
    assert float(np.abs(d_ranks.cpu().numpy().astype(np.float64) - o_at[0]).sum()) <= 1e-6
    # device top-k of the output
    ids, vals = sp.pagerank_top_k_device(d_ranks, 20)
    h_ids, h_vals = sp.pagerank_top_k(d_ranks.cpu().numpy(), 20)
    assert np.array_equal(vals, h_vals) and np.array_equal(ids, h_ids)
    # max_iterations = 0: the initial, uniform vector
    rc, it0 = sp.pagerank_device_personalized(G.ptr, d_ranks, v, sp.make_pagerank_config(D, 1e-6, 0))[:2]
    assert rc == 0 and it0 == 0
    assert np.array_equal(d_ranks.cpu().numpy(), np.full(n, 1.0 / n, np.float32))  # n = 2^scale: 1/n and its sum are exact
    # the drop-in call: host ranks, literal fp32 normalisation
    A = sp.csr_from_arrays(n, n, rp, ci, va)
    assert sp.csr_to_gpu(A) == 0
    result, ranks = sp.pagerank_personalized(A, v, sp.make_pagerank_config(D, 1e-6, 100))
    assert abs(result.iterations - o_it) <= 1 and bool(result.converged) == o_conv
    assert float(np.abs(ranks.astype(np.float64) - orc_personalized(n, rp, ci, va, v, fixed_it=result.iterations)[0])
                 .sum()) <= 2e-6
    sp.pagerank_free(result)
    # personalization None is pagerank() itself
    r_none, ranks_none = sp.pagerank_personalized(A, None, sp.make_pagerank_config(D, 1e-6, 100))
    r_glob, ranks_glob = sp.pagerank(A, sp.make_pagerank_config(D, 1e-6, 100))
    assert r_none.iterations == r_glob.iterations and np.array_equal(ranks_none.view(np.uint32), ranks_glob.view(np.uint32))
    sp.pagerank_free(r_none)
    sp.pagerank_free(r_glob)
    sp.csr_destroy(A)


# --------------------------------------------------------------------------------------------- sharded ----
@pytest.mark.gpu
def test_sharded_object_set_and_clear(sp, orc, cuda):
    """A pr_dist handle (one rank): global ranks, then personalized, then cleared again -- the cleared run must give
    today's vector bit for bit, so the graphs captured with the personalization vector are not replayed."""
    import torch
    import gpu_spmv_b200.dist as Dm
    n, rp, ci, va = rmat(13, 8, 51)
    v = random_personalization(n, 51)
    csr = sp.DeviceCSR(n, n, torch.as_tensor(rp).to(cuda), torch.as_tensor(ci).to(cuda), torch.as_tensor(va).to(cuda))
    comm = Dm.NativeComm(0, 1, f"pprtest-{os.getpid()}")
    pr = Dm.NativeShardedPageRank(comm, csr, 0, n, Dm.EXCHANGE_P2P)
    try:
        def run():
            res = pr.run(D, 1e-6, 100)
            assert res.graph_replay == 1
            return res, pr.ranks(cuda).cpu().numpy().copy()
        res_a, a = run()
        pr.set_personalization(v)
        res_p, p = run()
        o = orc_personalized(n, rp, ci, va, v, fixed_it=res_p.iterations)[0]
        assert float(np.abs(p.astype(np.float64) - o).sum()) <= 1e-6
        assert float(np.abs(p.astype(np.float64) - a).sum()) > 1e-3  # the vector took effect
        pr.set_personalization(None)
        res_b, b = run()
        assert res_b.iterations == res_a.iterations and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    finally:
        pr.close()
        comm.close()
    # the constructor argument
    pr = Dm.NativeShardedPageRank(Dm.NativeComm(0, 1, f"pprtest2-{os.getpid()}"), csr, 0, n, Dm.EXCHANGE_P2P,
                                  personalization=v)
    try:
        res = pr.run(D, 1e-6, 100)
        assert res.iterations == res_p.iterations
        assert np.array_equal(pr.ranks(cuda).cpu().numpy().view(np.uint32), p.view(np.uint32))
    finally:
        pr.close()
        pr.comm.close()


@pytest.mark.gpu
def test_sharded_null_vector_is_pagerank_multi(sp, cuda):
    """spmv_b200_pagerank_multi_personalized with NULL is spmv_b200_pagerank_multi, bit for bit (2 ranks, one GPU)."""
    import gpu_spmv_b200.dist as Dm
    n, rp, ci, va = rmat(12, 8, 52)
    A = sp.csr_from_arrays(n, n, rp, ci, va)
    cfg = sp.make_pagerank_config(D, 1e-6, 100)
    devices = (C.c_int * 2)(0, 0)
    a, b = np.empty(n, np.float32), np.empty(n, np.float32)
    ra, rb = Dm.PrDistResult(), Dm.PrDistResult()
    assert sp.lib.spmv_b200_pagerank_multi(A, C.byref(cfg), 2, devices, 1, 4, 0, a.ctypes.data_as(C.c_void_p), C.byref(ra)) == 0
    assert sp.lib.spmv_b200_pagerank_multi_personalized(A, C.byref(cfg), None, 2, devices, 1, 4, 0,
                                                        b.ctypes.data_as(C.c_void_p), C.byref(rb)) == 0
    assert ra.iterations == rb.iterations and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    sp.csr_destroy(A)


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child(sys.argv[2])
