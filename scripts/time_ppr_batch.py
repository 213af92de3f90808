#!/usr/bin/env python
"""Batched personalized PageRank against single-vector runs, on one GPU.

    python scripts/time_ppr_batch.py [--scales 20,22,24,26] [--reps 5] [--k 8]

Graphs: R-MAT `scale` with edge factor 16 (bench.py's PageRank graphs).  k teleport vectors (seed sets of 64 nodes).
Per repeat, interleaved: one spmv_b200_pagerank_device_personalized run (vector 0) and one batch of all k vectors
(spmv_b200_pagerank_personalized_batch), both with tolerance 0, so both run exactly the given iteration count.  Each
is timed at K_LO and K_HI iterations and the difference over K_HI - K_LO is the time per iteration (set-up cancels);
the set-up is what remains of the K_LO run.  Prints ms per iteration, vector-iterations per second, the batch's
speed-up over k sequential single runs, the card's name and power limit, and checks that the batch's column 0 is
within L1 1e-6 of the single run at the same iteration count."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as S
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K_LO, K_HI = 4, 64


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scales", default="20,22,24,26")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--k", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is timed on the CPU")
    from _load_pkg import load_pkg
    sp = load_pkg()
    import gpu_spmv_b200.gen as gen
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    print(f"card: {card()}")
    k = args.k
    for scale in (int(s) for s in args.scales.split(",")):
        n, rp, ci, va = gen.rmat_pagerank_csr(scale, 16, 9, dev)
        G = sp.DeviceCSR(n, n, rp, ci, va)
        rng = np.random.default_rng(scale)
        seeds = np.sort(np.stack([rng.choice(n, 64, replace=False) for _ in range(k)]), axis=1)
        V = S.csr_matrix((rng.uniform(0.5, 2.0, k * 64).astype(np.float32), seeds.ravel(), np.arange(k + 1) * 64),
                         shape=(k, n))
        v0 = V[0].toarray().ravel()
        d_single = torch.empty(n, dtype=torch.float32, device=dev)

        def single(iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rc, it = sp.pagerank_device_personalized(G.ptr, d_single, v0, sp.make_pagerank_config(0.85, 0.0, iters))[:2]
            torch.cuda.synchronize()
            assert rc == 0 and it == iters, (rc, it)
            return time.perf_counter() - t0

        out = {}

        def batch(iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ranks, it = sp.pagerank_personalized_batch(G.ptr, V, sp.make_pagerank_config(0.85, 0.0, iters))[:2]
            torch.cuda.synchronize()
            assert (it == iters).all(), it
            out["ranks"] = ranks
            return time.perf_counter() - t0

        single(K_LO), batch(K_LO)  # warm-up: module load, first allocations
        per = {"single": [], "batch": []}
        setup = {"single": [], "batch": []}
        for _ in range(args.reps):
            for name, fn in (("single", single), ("batch", batch)):
                lo, hi = fn(K_LO), fn(K_HI)
                it_s = (hi - lo) / (K_HI - K_LO)
                per[name].append(it_s * 1e3)
                setup[name].append((lo - K_LO * it_s) * 1e3)
        # column 0 of the last batch (K_HI iterations) against a single run of the same length
        single(K_HI)
        l1 = float((out["ranks"][:, 0].double() - d_single.double()).abs().sum())
        med = {key: float(np.median(x)) for key, x in per.items()}
        nnz = G.struct.nnz
        print(f"R-MAT {scale} (n = {n}, nnz = {nnz}), k = {k}, {K_HI} vs {K_LO} iterations, "
              f"median of {args.reps} interleaved repeats:")
        for key, vecs in (("single", 1), ("batch", k)):
            x = per[key]
            print(f"  {key:6s} ms/iteration {med[key]:8.4f} (min {min(x):.4f}, max {max(x):.4f}), "
                  f"vector-iterations/s {vecs / med[key] * 1e3:10.1f}, set-up {float(np.median(setup[key])):.2f} ms")
        print(f"  batch vs {k} sequential single runs: {k * med['single'] / med['batch']:.2f}x vector throughput; "
              f"column 0 vs the single run: L1 {l1:.3e} ({'ok' if l1 <= 1e-6 else 'MISMATCH'})")
        del G, rp, ci, va, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
