#!/usr/bin/env python
"""ms per PageRank iteration, global against personalized, on one GPU.

    python scripts/time_personalized_pagerank.py [--scales 12,24,26] [--reps 5]

Graphs: R-MAT `scale` with edge factor 16 (bench.py's PageRank graphs); the personalization vector is a 1 % seed
set.  Global and personalized runs alternate, `reps` times each; the median and the range are printed with the
card's name and power limit.
- Large graphs (scale > 13) take the multi-kernel loop with the plan pr_plan_create picks for a whole graph
  (segmented stream or hub columns).  They run as a one-rank NativeShardedPageRank for FIXED iterations: its
  device_seconds are CUDA events around the graph-replayed loop only, so set-up and graph capture are excluded.
  set_personalization switches the form between runs.
- Small graphs take the one-kernel loop: spmv_b200_pagerank_device_personalized with tolerance 0 runs K_LO and K_HI
  iterations, and the time difference over K_HI - K_LO cancels the set-up."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K_LO, K_HI = 10, 2000  # one-kernel loop
FIXED = 50             # multi-kernel loop


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scales", default="12,24,26")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is timed on the CPU")
    from _load_pkg import load_pkg
    sp = load_pkg()
    import gpu_spmv_b200.gen as gen
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    print(f"card: {card()}")
    for scale in (int(s) for s in args.scales.split(",")):
        n, rp, ci, va = gen.rmat_pagerank_csr(scale, 16, 9, dev)
        G = sp.DeviceCSR(n, n, rp, ci, va)
        rng = np.random.default_rng(scale)
        v = np.zeros(n, np.float32)
        v[rng.choice(n, max(1, n // 100), replace=False)] = rng.uniform(0.5, 2.0, max(1, n // 100))
        if scale > 13:
            import gpu_spmv_b200.dist as D
            comm = D.NativeComm(0, 1, f"time-ppr-{os.getpid()}-{scale}")
            pr = D.NativeShardedPageRank(comm, G, 0, n, D.EXCHANGE_P2P)

            def run(vec):
                pr.set_personalization(vec)
                res = pr.run(0.85, 0.0, FIXED, fixed_iterations=FIXED)
                return res.device_seconds / res.iterations_launched * 1e3
        else:
            d_ranks = torch.empty(n, dtype=torch.float32, device=dev)

            def timed(vec, iters):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rc, it = sp.pagerank_device_personalized(G.ptr, d_ranks, vec, sp.make_pagerank_config(0.85, 0.0, iters))[:2]
                torch.cuda.synchronize()
                assert rc == 0 and it == iters, (rc, it)
                return time.perf_counter() - t0

            def run(vec):
                return (timed(vec, K_HI) - timed(vec, K_LO)) / (K_HI - K_LO) * 1e3

        for vec in (None, v):  # warm-up: module load, plans, graph capture
            run(vec)
        per = {"global": [], "personalized": []}
        for _ in range(args.reps):
            for name, vec in (("global", None), ("personalized", v)):
                per[name].append(run(vec))
        med = {k: float(np.median(x)) for k, x in per.items()}
        for k, x in per.items():
            print(f"R-MAT {scale} (n = {n}, nnz = {G.struct.nnz}) {k:13s} ms/iteration: median {med[k]:.4f}, "
                  f"min {min(x):.4f}, max {max(x):.4f} over {len(x)} interleaved repeats")
        print(f"R-MAT {scale} personalized / global: {med['personalized'] / med['global']:.4f}")
        if scale > 13:
            pr.close()
            comm.close()
        del G, rp, ci, va
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
