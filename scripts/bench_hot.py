#!/usr/bin/env python
"""Tuning aid: plain merge-path vs the planned kernels (csr_hot_kernels.cu, csr_seg_kernels.cu).

    python scripts/bench_hot.py --scale 24 --caps 0,32768,16384,4096 [--pagerank] [--relabelled]
    SPMV_B200_PLAN=seg python scripts/bench_hot.py --dataset c2 --caps 0

Prints one JSON line per measurement (CUDA events on the launching stream, after warm-up)."""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=24)
    ap.add_argument("--caps", default="0")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--pagerank", action="store_true")
    ap.add_argument("--relabelled", action="store_true")
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--dataset", default="rmat", choices=["rmat", "c2", "c3"])
    args = ap.parse_args()

    import numpy as np
    import torch
    import bench as B
    from _load_pkg import load_pkg
    sp = load_pkg()
    import gpu_spmv_b200.dist as D
    import gpu_spmv_b200.gen as gen

    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    peak, _ = B.measured_peak()
    stream = torch.cuda.Stream()
    s_ptr = stream.cuda_stream
    if args.dataset == "c2":
        n = 4096 * 4096
        rp, ci, va = gen.laplacian_2d_csr(4096, dev)
    elif args.dataset == "c3":
        n = 50_000_000
        rp, ci, va = gen.short_rows_with_outliers_csr(n, 43, dev)
    else:
        n, _, rp, ci, va, _ = gen.rmat_pagerank_shard(args.scale, 16, args.seed, 0, 1, dev, relabelled=args.relabelled)
    torch.cuda.synchronize()
    A = sp.DeviceCSR(n, n, rp, ci, va)
    x = gen.vector_pm1(n, 7, dev)
    y0 = torch.empty(n, dtype=torch.float32, device=dev)
    y1 = torch.empty(n, dtype=torch.float32, device=dev)
    nbytes = sp.csr_bytes(n, n, ci.numel())
    cfg = sp.make_config(sp.MERGE_PATH)

    def emit(**kw):
        print(json.dumps(kw), flush=True)

    def plain():
        assert sp.lib.spmv_b200_spmv_csr_async(A.ptr, sp.dptr(x), sp.dptr(y0), C.byref(cfg), C.c_void_p(s_ptr)) == 0

    r = B.bench_kernel(torch, sp, stream, plain, nbytes, args.steps, 3)
    emit(what="plain merge-path", dataset=args.dataset, scale=args.scale, relabelled=args.relabelled, ms=r["ms_per_step"], gbs=r["gbs"],
         frac_of_measured_peak=r["gbs"] / peak, frac_of_8000=r["gbs"] / 8000.0)

    for cap in [int(c) for c in args.caps.split(",")]:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plan = sp.CsrPlan(A.ptr, cap, force=args.dataset != "rmat")
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        n_hot, hot_nnz, mode = plan.info()

        def hot():
            assert plan.spmv(x, y1, s_ptr) == 0

        r = B.bench_kernel(torch, sp, stream, hot, nbytes, args.steps, 3)
        torch.cuda.synchronize()
        same = bool(torch.equal(y0.view(torch.int32), y1.view(torch.int32)))
        emit(what="planned kernel (%s)" % os.environ.get("SPMV_B200_PLAN", "seg"), cap=cap, hot_columns=n_hot, hot_nnz_frac=hot_nnz / max(ci.numel(), 1), mode=mode,
             plan_build_ms=build_ms, ms=r["ms_per_step"], gbs=r["gbs"], frac_of_measured_peak=r["gbs"] / peak,
             frac_of_8000=r["gbs"] / 8000.0, bit_identical_to_plain=same)
        plan.close()

    if args.pagerank:
        shard = D.CudaShard(n, 0, rp, ci, va, stream=s_ptr)
        shard.damping = 0.85
        with torch.cuda.stream(stream):
            shard.setup_dangling()
        iters = 20
        for cap in (0, -1):
            used = shard.set_hot(cap)
            with torch.cuda.stream(stream):
                r_a = torch.empty(n, dtype=torch.float32, device=dev)
                r_b = torch.empty_like(r_a)
                partial = torch.zeros(3, dtype=torch.float64, device=dev)
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                shard.init_vector(r_a)
                for it in range(3 + iters):
                    if it == 3:  # after 3 warm-up steps, time `iters` steps from the start vector
                        shard.init_vector(r_a)
                        t0.record()
                    shard(r_a, r_b, partial)
                    shard.dsum.copy_(partial[2:3].to(torch.float32))  # the dangling mass of the vector just written
                    r_a, r_b = r_b, r_a
                t1.record()
                torch.cuda.synchronize()
                ms = t0.elapsed_time(t1) / iters
            residual = float(np.sqrt(np.float32(partial[0].item())))
            emit(what="pagerank", hot_columns=used, ms_per_iter=ms, iters_per_s=1e3 / ms, residual=residual,
                 checksum=float(r_a.double().sum().item()), effective_gbs=nbytes / (ms * 1e-3) / 1e9)
        shard.close()


if __name__ == "__main__":
    main()
