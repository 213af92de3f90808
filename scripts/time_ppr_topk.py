#!/usr/bin/env python
"""Per-seed top-K personalized PageRank against the dense batch, on one GPU.

    python scripts/time_ppr_topk.py [--scales 20,22,24] [--reps 3] [--k 64] [--top 100] [--wall-iters 10]

Graphs: R-MAT `scale` with edge factor 16 (bench.py's PageRank graphs).  k teleport vectors (seed sets of 64 nodes),
tolerance 0, so every run does exactly the given iteration count.  Per graph, interleaved repeats of:
  dense  spmv_b200_pagerank_personalized_batch, the [n][k] rank matrix;
  top-K  spmv_b200_pagerank_personalized_batch_top_k, each column's `top` best nodes;
each at K_LO and K_HI iterations.  Reported:
  (a) one iteration of one chunk of 8 columns (dense, (K_HI - K_LO) difference) next to the selection of one chunk,
      taken as (top-K - dense) at the same iteration count over the k / 8 chunks: the selection's cost minus the
      dense path's scale into [n][k];
  (b) one top-K call against what a caller does without it: the dense batch, then pagerank_top_k_device on each
      ranks[:, c].contiguous() (K_HI iterations both);
  (c) R-MAT 20 with one-hot seeds and k such that n * k * 4 bytes exceed the device's memory (--wall-iters
      iterations): time and seeds per second.
Every top-K run is checked against the dense batch: row 0 must equal the top of column 0 bit for bit.  Prints the
card's name and power limit."""
import argparse
import math
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as S
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K_LO, K_HI = 4, 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def top_of(col, top):
    """(ids, value bits) of the `top` best entries of a host column: rank descending, id ascending."""
    order = np.lexsort((np.arange(col.size), -col))[:top]
    return order.astype(np.int32), col[order].view(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scales", default="20,22,24")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--top", type=int, default=100)
    ap.add_argument("--wall-iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is timed on the CPU")
    from _load_pkg import load_pkg
    sp = load_pkg()
    import gpu_spmv_b200.gen as gen
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    print(f"card: {card()}")
    k, top = args.k, args.top
    chunks = (k + 7) // 8
    cfg = lambda iters: sp.make_pagerank_config(0.85, 0.0, iters)  # noqa: E731

    for scale in (int(s) for s in args.scales.split(",")):
        n, rp, ci, va = gen.rmat_pagerank_csr(scale, 16, 9, dev)
        G = sp.DeviceCSR(n, n, rp, ci, va)
        rng = np.random.default_rng(scale)
        seeds = np.sort(np.stack([rng.choice(n, 64, replace=False) for _ in range(k)]), axis=1)
        V = S.csr_matrix((rng.uniform(0.5, 2.0, k * 64).astype(np.float32), seeds.ravel(), np.arange(k + 1) * 64),
                         shape=(k, n))
        ok = True

        def dense(iters):
            return sp.pagerank_personalized_batch(G.ptr, V, cfg(iters))[0]

        def topk(iters):
            return sp.pagerank_personalized_batch_top_k(G.ptr, V, top, cfg(iters))[:2]

        def today(iters):
            ranks = dense(iters)
            return [sp.pagerank_top_k_device(ranks[:, c].contiguous(), top) for c in range(k)]

        def check(ranks, ids, vals):
            e_ids, e_bits = top_of(ranks[:, 0].cpu().numpy(), top)
            return (np.array_equal(ids[0].cpu().numpy(), e_ids) and
                    np.array_equal(vals[0].cpu().numpy().view(np.uint32), e_bits))

        dense(K_LO), topk(K_LO), today(K_LO)  # warm-up: module loads, first allocations
        t = {key: [] for key in ("dense_lo", "dense_hi", "topk_lo", "topk_hi", "today_hi")}
        for _ in range(args.reps):
            t["dense_lo"].append(timed(lambda: dense(K_LO))[0])
            t["topk_lo"].append(timed(lambda: topk(K_LO))[0])
            s, ranks = timed(lambda: dense(K_HI))
            t["dense_hi"].append(s)
            s, (ids, vals) = timed(lambda: topk(K_HI))
            t["topk_hi"].append(s)
            ok &= check(ranks, ids, vals)
            del ranks
            t["today_hi"].append(timed(lambda: today(K_HI))[0])
        med = {key: float(np.median(x)) * 1e3 for key, x in t.items()}
        it_chunk = (med["dense_hi"] - med["dense_lo"]) / (K_HI - K_LO) / chunks
        sel = [(tk - d) / chunks for tk, d in ((med["topk_lo"], med["dense_lo"]), (med["topk_hi"], med["dense_hi"]))]
        print(f"R-MAT {scale} (n = {n}, nnz = {G.struct.nnz}), k = {k} seed sets of 64, top = {top}, "
              f"median of {args.reps} interleaved repeats:")
        print(f"  (a) one iteration of one chunk {it_chunk:8.3f} ms; selection of one chunk (top-K - dense, per chunk) "
              f"{sel[0]:.3f} ms at {K_LO} iterations, {sel[1]:.3f} ms at {K_HI}")
        print(f"  (b) {K_HI} iterations: top-K call {med['topk_hi']:9.1f} ms; dense batch {med['dense_hi']:9.1f} ms + "
              f"{k} x pagerank_top_k_device = {med['today_hi']:9.1f} ms ({med['today_hi'] / med['topk_hi']:.2f}x)")
        print(f"      dense output {n * k * 4 / 2**30:.2f} GiB, top-K output {k * top * 8 / 2**20:.2f} MiB; "
              f"row 0 vs the dense column: {'bit-identical' if ok else 'MISMATCH'}")
        del G, rp, ci, va, V
        torch.cuda.empty_cache()

    # (c) past the memory wall: more one-hot seeds than a dense n x k output could hold
    n, rp, ci, va = gen.rmat_pagerank_csr(20, 16, 9, dev)
    G = sp.DeviceCSR(n, n, rp, ci, va)
    total = torch.cuda.mem_get_info()[1]
    kw = math.ceil(1.05 * total / (4 * n))
    seeds = (np.arange(kw, dtype=np.int64) * 7919) % n
    sp.pagerank_personalized_batch_top_k(G.ptr, seeds[:8], top, cfg(args.wall_iters))  # warm-up
    s, (ids, vals, it) = timed(lambda: sp.pagerank_personalized_batch_top_k(G.ptr, seeds, top, cfg(args.wall_iters))[:3])
    pick = [0, kw // 2, kw - 1]
    ranks = sp.pagerank_personalized_batch(G.ptr, seeds[pick], cfg(args.wall_iters))[0].cpu().numpy()
    ok = all(np.array_equal(ids[c].cpu().numpy(), top_of(ranks[:, j], top)[0]) and
             np.array_equal(vals[c].cpu().numpy().view(np.uint32), top_of(ranks[:, j], top)[1])
             for j, c in enumerate(pick))
    print(f"(c) R-MAT 20 (n = {n}, nnz = {G.struct.nnz}), k = {kw} one-hot seeds (dense output {kw * n * 4 / 1e9:.1f} GB, "
          f"device memory {total / 1e9:.1f} GB), top = {top}, {args.wall_iters} iterations: {s:.2f} s, "
          f"{kw / s:.0f} seeds/s; "
          f"rows 0, k/2, k-1 vs the dense batch of those seeds: {'bit-identical' if ok else 'MISMATCH'}")


if __name__ == "__main__":
    main()
