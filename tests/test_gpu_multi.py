"""Sharded PageRank on >= 2 GPUs of one box: the NCCL transport, the fused peer-store exchange and the
fused NVSwitch-multicast exchange must all reproduce the f64 oracle, and must be bitwise identical to each
other (same kernels, same summation order, only the transport differs).
Skipped on boxes with a single GPU."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_native_pagerank_multi_transports_bit_identical(sp, orc, cuda):
    """spmv_b200_pagerank_multi on the GPUs of the box (one process, one host thread per device): multicast,
    peer stores and NCCL must give bit-identical vectors, within L1 1e-6 of the f64 oracle restatement, for
    10 fixed iterations and for runs to convergence (tolerance 1e-6, at most 100 iterations), where every
    transport must also stop at the oracle's iteration."""
    import ctypes as C
    import gpu_spmv_b200.dist as D
    import gpu_spmv_b200.gen as gen
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    for scale, tol, fixed in ((18, 0.0, 10), (14, 1e-6, 0), (18, 1e-6, 0)):
        n, rp, ci, va = gen.rmat_pagerank_csr(scale, 16, 7, "cpu")
        rp_n, ci_n, va_n = rp.numpy(), ci.numpy(), va.numpy()
        A = sp.csr_from_arrays(n, n, rp_n, ci_n, va_n)
        cfg = sp.make_pagerank_config(0.85, tol, fixed or 100)
        o_ranks, o_it, _, _, o_conv = orc.pagerank_f64(n, n, rp_n, ci_n, va_n, 0.85, 1e-6, 100, fixed_it=fixed)
        assert fixed or o_conv
        results = {}
        for name, exchange in (("auto", D.EXCHANGE_AUTO), ("p2p", D.EXCHANGE_P2P), ("nccl", D.EXCHANGE_NCCL)):
            ranks = np.empty(n, np.float32)
            res = D.PrDistResult()
            rc = sp.lib.spmv_b200_pagerank_multi(A, C.byref(cfg), world, None, exchange, 4, fixed,
                                                 ranks.ctypes.data_as(C.c_void_p), C.byref(res))
            assert rc == 0, (name, sp.spmv_error_string(rc))
            assert res.iterations == (fixed or o_it), (scale, name, res.iterations, o_it)
            if not fixed:
                assert res.converged == 1, (scale, name)
            assert float(np.abs(ranks.astype(np.float64) - o_ranks.astype(np.float64)).sum()) <= 1e-6, (scale, name)
            results[name] = (ranks, (res.iterations, res.final_residual, res.converged), res.exchange)
        print(f"scale {scale}, fixed {fixed}: transports used:", {k: D.EXCHANGE_NAMES[v[2]] for k, v in results.items()})
        for name in ("p2p", "nccl"):
            assert results[name][1] == results["auto"][1], (scale, name, results[name][1], results["auto"][1])
            assert np.array_equal(results["auto"][0].view(np.uint32), results[name][0].view(np.uint32)), (scale, name)
        sp.csr_destroy(A)


def test_plain_c_caller_of_the_multi_gpu_entry_point(cuda):
    """tests/c/pagerank_multi_test.c: a C program linked against libspmv_b200.so, no Python in the loop."""
    import subprocess
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "c", "_build", "pagerank_multi_test")
    if not os.path.exists(exe):
        pytest.skip("tests/c/_build/pagerank_multi_test not built (run __graft_entry__.build())")
    for exchange in ("-1", "1", "0"):
        p = subprocess.run([exe, "2", "16", exchange], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert p.returncode == 0 and "PASS" in p.stdout, p.stdout[-2000:]
