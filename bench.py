#!/usr/bin/env python
"""bench.py -- headline benchmark of the SpMV hot path (see BASELINE.json / BASELINE.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--quick] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Every timed SpMV loop runs exactly K steps (PageRank runs --pr-iters iterations).
--dump-outputs DIR writes, after the timed steps, what each timed path computed in
its last step as DIR/<name>.npy (float32, rank 0): every SpMV kernel, plan and
host-buffer call timed on configs 2, 3 and 4, and every PageRank vector timed
(one per graph: the transports are checked bit-identical).  Each file is the same
seeded sample of DUMP_ROWS entries of its vector, so that two builds can be
compared output for output on identical inputs.  The reference arm writes its
config-2 y under the same name and sample (the positions inside its band).

A "step" is one pass of the hot path over one batch of synthetic input: one
ELL SpMV over BASELINE config 2 (5-point Laplacian on a 4096^2 grid, 16.7 M
rows, 83.9 M non-zeros, 805 MB of matrix -- larger than L2, so no flush is
needed between iterations).  `value` is whole-job effective HBM GB/s =
algorithmic bytes (reference src/bandwidth.cpp:66-75) x steps / device time,
inputs resident in HBM.  `e2e` is the same metric through the reference-facing
C-ABI call that takes HOST x / y buffers (spmv_b200_spmv_ell_host: H2D of x,
the product and the way down of y overlapped -- one persistent kernel consumes x
as the upload lands and stores y into the pinned host buffer --, all inside the
timed region).

BASELINE.json's metric has a second half -- PageRank iterations/s at 1/2/4/8
GPUs on R-MAT 26 -- and a sharded SpMV case (config 4, R-MAT 24 merge-path).
Both are measured in the same run and reported as TOP-LEVEL scalars of the
line (`pagerank_iters_per_s`, `pagerank_ms_per_iter`, `pagerank_exchange`,
`pagerank_1gpu_iters_per_s`, `pagerank_speedup_vs_1gpu`, `rmat24_merge_frac`,
`config2_csr_frac`, ...), with the details under `extra`.  The sharded
PageRank runs through the native C++ path (spmv_b200_pr_dist_*: strong
scaling, one graph split over the N ranks); before it is timed, `parity`
checks it against the CPU oracle (scale-20 graph, every transport, 10 fixed
iterations, L1 <= 1e-6, transports bit-identical) and, at full size, that every
rank holds the bit-identical vector with sum 1 -- a mismatch makes the run fail.

N > 1 (one rank per GPU): weak scaling for the headline -- every rank owns a
16.7 M-row band (row shard) of a 4096 x (4096 N) Laplacian with the vector
replicated, no data-path collective.

--impl reference times the reference's own CPU implementation of the step
(spmv_cpu_ell from oracle/_ref, the unmodified reference sources; the oracle
port if that library is absent) on the host, rank 0 only.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = 4096            # BASELINE config 2
SEED_X = 42
FALLBACK_PEAK_GBS = 6650.0
DUMP_ROWS = 1 << 19    # --dump-outputs: entries kept per output vector (15 vectors at most: 30 MiB)
DUMP_SEED = 2024


def dump_index(n):
    """The sorted positions of an n-vector that --dump-outputs keeps: all of them, or a fixed seeded sample."""
    import numpy as np
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))


def write_outputs(directory, outputs):
    """--dump-outputs: each float32 array of `outputs` as <directory>/<name>.npy."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float32))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return FALLBACK_PEAK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- reference arm

WORKLOAD = ("config2: 5-point Laplacian 4096x4096 grid per GPU (16.7M rows, 83.9M nnz), ELL width 5, spmv_ell; "
            "x = hash U[-1,1)")


def headline_config(rows, nnz, bytes_per_step, world):
    """`config` of the JSON line -- the same keys and strings in both arms (same_config at N = 1)."""
    return {"workload": WORKLOAD, "rows": rows, "nnz": nnz, "bytes_per_step": bytes_per_step,
            "l2": "inputs (805 MB per GPU) larger than L2 / LLC, no flush",
            "parallelism": f"row shards x{world}, x replicated"}


def standalone_gen():
    """gpu-spmv_b200/gen.py loaded as a plain module (pure torch): the reference arm must not load the
    product package, whose import pulls in libspmv_b200.so."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("spmv_bench_gen", os.path.join(ROOT, "gpu-spmv_b200", "gen.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build_config2_host(rows_lo, rows_hi, grid_y):
    """Config-2 band as host CSR arrays + x, generated on the CPU (no product code involved)."""
    gen = standalone_gen()
    rp, ci, va = gen.laplacian_band_csr(GRID, rows_lo, rows_hi, grid_y, "cpu")
    x = gen.vector_pm1(GRID * grid_y, SEED_X, "cpu").numpy()
    return rp.numpy(), ci.numpy(), va.numpy(), x


def cpu_reference_time(rp, ci, va, x, rows, cols, reps):
    """Seconds per spmv_cpu_ell pass through the unmodified reference (oracle/_ref), else the
    oracle port.  Returns (seconds, kind, threads, y of the last pass)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_binding import Oracle, Ref
    if Ref.available():
        ref = Ref()
        h, keep = ref.csr_wrap(rows, cols, rp, ci, va)
        he, st = ref.ell_from_csr(h)
        assert st == 0
        y = np.empty(rows, np.float32)
        fp = C.POINTER(C.c_float)
        ref.L.ref_time_spmv_cpu_ell(he, x.ctypes.data_as(fp), y.ctypes.data_as(fp), 1)  # warm-up
        sec = ref.L.ref_time_spmv_cpu_ell(he, x.ctypes.data_as(fp), y.ctypes.data_as(fp), reps)
        ref.L.ref_ell_destroy(he)
        ref.L.ref_csr_destroy(h)
        return sec, "reference", 1, y
    orc = Oracle()
    w, ec, ev = orc.ell_from_csr(rows, rp, ci, va)
    orc.spmv_ell(rows, w, ec, ev, x)
    t0 = time.perf_counter()
    for _ in range(reps):
        y = orc.spmv_ell(rows, w, ec, ev, x)
    return (time.perf_counter() - t0) / reps, "port", 1, y


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_full = GRID * GRID
    # bounded sample: a probe band sizes the per-step sample so that steps + warm-up stay near 2 minutes
    probe_rows = 1 << 20
    rp, ci, va, x = build_config2_host(0, probe_rows, GRID)
    probe_sec, _, _, _ = cpu_reference_time(rp, ci, va, x, probe_rows, n_full, 2)
    budget_rows = int(120.0 / max(args.steps + args.warmup, 1) / (probe_sec / probe_rows))
    n = max(probe_rows, min(n_full, budget_rows // GRID * GRID))
    rp, ci, va, x = build_config2_host(0, n, GRID)
    bytes_step = 8 * n * 5 + 4 * (n_full if n == n_full else n + GRID) + 4 * n
    for _ in range(max(args.warmup, 1) - 1):
        cpu_reference_time(rp, ci, va, x, n, n_full, 1)
    sec, kind, threads, y = cpu_reference_time(rp, ci, va, x, n, n_full, args.steps)
    if args.dump_outputs is not None:
        idx = dump_index(n_full)  # the GPU arm's sample of config-2 y; a band keeps the positions inside it
        write_outputs(args.dump_outputs, {"config2_ell_y": y[idx[idx < n]]})
    gbs = bytes_step / sec / 1e9
    sample = ("the full config-2 matrix" if n == n_full else f"the first {n} rows (a band) of the config-2 matrix")
    line = {
        "impl": "reference", "metric": "spmv_effective_hbm_gbs", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(n, 5 * n - 4 * GRID if n == n_full else 5 * n - 2 * (n // GRID) - GRID, bytes_step, 1),
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": kind,
                         "sample": f"{sample}, {args.steps} passes of spmv_cpu_ell per run, one pass per step "
                                   "(single-threaded: the reference has no threading)"},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- product arm

def timed_region(torch, stream, fn, steps, dist_on):
    """K calls of fn on `stream` between two CUDA events, barrier + sync on both sides."""
    import torch.distributed as dist
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        start.record(stream)
        for _ in range(steps):
            fn()
        stop.record(stream)
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    ms = start.elapsed_time(stop)
    if dist_on:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def bench_kernel(torch, sp, stream, launch, bytes_per_launch, steps, warmup, dist_on=False, world=1):
    torch.cuda.synchronize()  # inputs were produced on torch's default stream; `stream` does not wait for it
    for _ in range(max(warmup, 3)):
        launch()
    torch.cuda.synchronize()
    ms = timed_region(torch, stream, launch, steps, dist_on)
    per = ms / steps
    return {"ms_per_step": per, "gbs": world * bytes_per_launch / (per * 1e-3) / 1e9}


def ncu_traffic_for(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_name` from the committed
    `ncu --set full` raw page (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py from the
    capture; keyed by kernel name and by the hash of the kernel's source file, so a stale capture
    reads as null instead of a wrong number)."""
    import hashlib
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            table = json.load(f)
        entry = table[kernel_name]
        with open(os.path.join(ROOT, entry["source"]), "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()[:16]
        if digest != entry["source_sha256_16"]:
            return None, f"stale: {entry['source']} changed since {entry['capture']}"
        return float(entry["dram_bytes_per_launch"]), entry["capture"]
    except Exception as exc:  # no table, no entry: unknown
        return None, f"unavailable ({type(exc).__name__})"


def nvlink_bytes(index):
    """(tx, rx) payload bytes moved over all NVLinks of GPU `index` so far, or None when the driver does not
    count them: NVML field values NVLINK_THROUGHPUT_DATA_TX / _RX summed over the links (KiB units), else
    `nvidia-smi nvlink -gt d`."""
    import re
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        tx_id = getattr(pynvml, "NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX", 138)
        rx_id = getattr(pynvml, "NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX", 139)
        vals = pynvml.nvmlDeviceGetFieldValues(h, [(tx_id, 0xFFFFFFFF), (rx_id, 0xFFFFFFFF)])  # scope: all links
        out = []
        for v in vals:
            if v.nvmlReturn != 0:
                raise RuntimeError("field not supported")
            out.append(int(v.value.ullVal) * 1024)
        if out[0] or out[1]:
            return out[0], out[1]
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], capture_output=True, text=True,
                             timeout=20).stdout
    except Exception:
        return None
    tx = sum(int(v) for v in re.findall(r"Data Tx:\s*(\d+)\s*KiB", out))
    rx = sum(int(v) for v in re.findall(r"Data Rx:\s*(\d+)\s*KiB", out))
    if not re.search(r"Data Tx", out) or (tx == 0 and rx == 0):
        return None  # counters absent or not maintained on this box
    return tx * 1024, rx * 1024


def vector_checksum(torch, v):
    """Two 64-bit integer checksums of the bit pattern of a float32 device vector (order-sensitive)."""
    bits = v.view(torch.int32).to(torch.int64)
    idx = torch.arange(bits.numel(), dtype=torch.int64, device=v.device) % 1000003 + 1
    return int(bits.sum().item()), int((bits * idx).sum().item())


def run_product_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from _load_pkg import load_pkg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    # stdout carries exactly ONE JSON line: whatever libraries print while the benchmark runs (NCCL writes its
    # version banner with printf) goes to stderr; the real stdout is restored for the line at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_on = world > 1
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    sp = load_pkg()
    import gpu_spmv_b200.dist as D
    import gpu_spmv_b200.gen as gen

    peak, peak_src = measured_peak()
    stream = torch.cuda.Stream()
    s_ptr = stream.cuda_stream
    extra = {}
    scalars = {}
    parity = {}
    session = f"bench-{os.environ.get('MASTER_PORT', '0')}-{os.environ.get('TORCHELASTIC_RUN_ID', 'x')}-{os.getppid() if dist_on else os.getpid()}"
    comm = D.NativeComm(rank, world, session) if dist_on else None

    def log(msg):
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    def max_over_ranks(v):
        if not dist_on:
            return float(v)
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(flag):
        if not dist_on:
            return bool(flag)
        t = torch.tensor([1.0 if flag else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() == 1.0)

    def r4(v):
        return float(f"{v:.5g}")

    outputs = {}

    def keep_output(name, v):
        """--dump-outputs: the sample of vector v (device or host) that is written as <name>.npy at the end."""
        if args.dump_outputs is not None and rank == 0:
            idx = torch.from_numpy(dump_index(v.numel())).to(v.device)
            outputs[name] = v[idx].cpu().numpy().astype(np.float32)

    # ---- headline: config 2, ELL, one 16.7 M-row band per rank (weak scaling) -----------------
    log("config 2: build + ELL headline")
    n_loc = GRID * GRID
    grid_y = GRID * world
    n_cols = GRID * grid_y
    rp, ci, va = gen.laplacian_band_csr(GRID, rank * n_loc, (rank + 1) * n_loc, grid_y, dev)
    A = sp.DeviceCSR(n_loc, n_cols, rp, ci, va)
    E = sp.ell_create(0, 0, 0)
    assert sp.ell_from_csr_device(E, A.ptr) == 0 and E.contents.max_nnz_per_row == 5
    x = gen.vector_pm1(n_cols, SEED_X, dev)
    y = torch.empty(n_loc, dtype=torch.float32, device=dev)
    x_touched = n_loc + 2 * GRID if world > 1 else n_cols   # a band only reads its rows +- one grid line of x
    ell_bytes = 8 * n_loc * 5 + 4 * x_touched + 4 * n_loc
    csr_bytes = 8 * ci.numel() + 4 * (n_loc + 1) + 4 * x_touched + 4 * n_loc
    nnz_total = 5 * n_loc * world - 2 * GRID - 2 * GRID * world

    def ell_step():
        rc = sp.lib.spmv_b200_spmv_ell_async(E, sp.dptr(x), sp.dptr(y), C.c_void_p(s_ptr))
        assert rc == 0

    torch.cuda.synchronize()  # x / matrix were produced on the default stream; `stream` does not wait for it
    for _ in range(max(args.warmup, 3)):
        ell_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches_before = sp.launch_count()
    ms = timed_region(torch, stream, ell_step, args.steps, dist_on)
    gpu_launches = sp.launch_count() - launches_before
    y_device_path = y.clone()
    torch.cuda.synchronize()  # the clone runs on the default stream, the load phase below rewrites y on `stream`
    keep_output("config2_ell_y", y_device_path)
    # untimed: keep the GPU under the same load for ~400 ms so the clock sampler sees it loaded
    if ms < 400:
        for _ in range(int(400 / max(ms / args.steps, 1e-3)) + 1):
            ell_step()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_per_step = ms / args.steps
    value = world * ell_bytes / (ms_per_step * 1e-3) / 1e9
    launch_gbs = ell_bytes / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: the C-ABI call that takes HOST x / y (pinned); H2D, kernel, D2H inside the timed region ---
    log("e2e")
    x_host = x.cpu().pin_memory()
    y_host = torch.empty(n_loc, dtype=torch.float32).pin_memory()
    res = sp.SpMVResult()

    def e2e_serial_step():  # what a caller of the reference writes: cudaMemcpy up, spmv_ell, cudaMemcpy down
        x.copy_(x_host, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        rc = sp.lib.spmv_b200_spmv_ell(E, sp.dptr(x), sp.dptr(y), None, n_cols, C.byref(res))
        assert rc == 0
        y_host.copy_(y, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    host_plan = C.c_void_p()
    assert sp.lib.spmv_b200_ell_host_plan_create(E, 0, C.byref(host_plan)) == 0
    h2d_bytes, d2h_bytes = C.c_ulonglong(0), C.c_ulonglong(0)
    assert sp.lib.spmv_b200_ell_host_plan_bytes(host_plan, C.byref(h2d_bytes), C.byref(d2h_bytes)) == 0
    c_gated, c_down = C.c_int(0), C.c_int(0)
    assert sp.lib.spmv_b200_ell_host_plan_gated(host_plan, C.byref(c_gated), C.byref(c_down)) == 0

    def e2e_step():  # blocking: returns when y_host is complete
        rc = sp.lib.spmv_b200_spmv_ell_host(host_plan, x_host.data_ptr(), y_host.data_ptr())
        assert rc == 0

    def wall_time(fn, steps):
        for _ in range(max(3, args.warmup)):  # untimed: the first copies out of freshly pinned pages are slow
            fn()
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return max_over_ranks((time.perf_counter() - t0) / steps)

    y_host.zero_()
    e2e_sec = wall_time(e2e_step, args.steps)
    e2e_same = bool(torch.equal(y_host.view(torch.int32), y_device_path.cpu().view(torch.int32)))
    keep_output("config2_ell_host_y", y_host)
    serial_sec = wall_time(e2e_serial_step, args.steps)
    keep_output("config2_ell_host_serial_y", y_host)
    # still gated after the timed calls (a call whose x did not arrive in time would have fallen back for good)
    assert sp.lib.spmv_b200_ell_host_plan_gated(host_plan, C.byref(c_gated), None) == 0
    host_gated = bool(c_gated.value)
    sp.lib.spmv_b200_ell_host_plan_destroy(host_plan)
    e2e = {"value": world * ell_bytes / e2e_sec / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(h2d_bytes.value) * world,
           "d2h_bytes_per_step": int(d2h_bytes.value) * world, "ms_per_step": e2e_sec * 1e3,
           "api": "spmv_b200_spmv_ell_host (blocking C ABI, pinned host x -> pinned host y; " + (
               "gated form: one upload copy over a sentinel-filled x, one persistent kernel that consumes x as it lands and stores y "
               "straight into the pinned host buffer)"
               if host_gated else "H2D / kernel / D2H pipelined over row chunks on three streams)"),
           "bit_identical_to_device_path": e2e_same,
           "serial_ms_per_step": serial_sec * 1e3}
    parity["e2e_host_call_bit_identical"] = e2e_same

    # ---- CPU baseline (rank 0, N = 1): the reference's spmv_cpu_ell on the same matrix; its y is the parity check
    log("cpu baseline")
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        reps = 3
        sec, kind, threads, y_cpu = cpu_reference_time(rp.cpu().numpy(), ci.cpu().numpy(), va.cpu().numpy(),
                                                       x_host.numpy(), n_loc, n_cols, reps)
        same = bool(np.array_equal(y_cpu.view(np.uint32), y_device_path.cpu().numpy().view(np.uint32)))
        parity["config2_ell_bit_identical_to_cpu_" + kind] = same
        cpu_baseline = {"value": ell_bytes / sec / 1e9, "unit": "GB/s", "cores": threads, "kind": kind,
                        "ms_per_step": sec * 1e3, "host_cpus": os.cpu_count(), "parity_checked": same,
                        "sample": f"the full config-2 matrix, {reps} passes of spmv_cpu_ell after 1 warm-up "
                                  "(single-threaded: the reference has no threading)"}

    # ---- extra: the CSR kernels on config 2 (the selector sends this matrix to VECTOR_CSR) --------------
    if not args.quick and not args.only_pagerank and world == 1:
        log("config 2: CSR kernels")
        for kernel, name in ((sp.VECTOR_CSR, "csr_vector"), (sp.SCALAR_CSR, "csr_scalar"), (sp.MERGE_PATH, "csr_merge")):
            cfg = sp.make_config(kernel)
            r = bench_kernel(torch, sp, stream, lambda: sp.lib.spmv_b200_spmv_csr_async(
                A.ptr, sp.dptr(x), sp.dptr(y), C.byref(cfg), C.c_void_p(s_ptr)), csr_bytes, args.steps, args.warmup,
                dist_on, world)
            torch.cuda.synchronize()
            keep_output(f"config2_{name}_y", y)
            entry = {"gbs": r4(r["gbs"]), "ms": r4(r["ms_per_step"]), "frac": r4(r["gbs"] / world / peak),
                     "frac_of_8000": r4(r["gbs"] / world / 8000.0)}
            if kernel != sp.MERGE_PATH:  # sequential order: bit-identical to the ELL result (= spmv_cpu_*)
                entry["bit_identical_to_ell"] = bool(torch.equal(y.view(torch.int32), y_device_path.view(torch.int32)))
                parity[f"config2_{name}_bit_identical"] = entry["bit_identical_to_ell"]
            extra[f"config2_{name}"] = entry
        scalars["config2_csr_frac"] = extra["config2_csr_vector"]["frac"]
        scalars["config2_csr_ms"] = extra["config2_csr_vector"]["ms"]
        # the same matrix through a CSR plan: no hub worth a table, >= 4 non-zeros per row -> the
        # segmented-stream kernel (csr_seg_kernels.cu)
        plan2 = sp.CsrPlan(A.ptr)
        r = bench_kernel(torch, sp, stream, lambda: plan2.spmv(x, y, s_ptr), csr_bytes, args.steps, args.warmup, dist_on, world)
        keep_output("config2_csr_planned_y", y)
        extra["config2_csr_planned"] = {"gbs": r4(r["gbs"]), "ms": r4(r["ms_per_step"]), "frac": r4(r["gbs"] / world / peak),
                                        "plan_mode": plan2.info()[2]}
        plan2.close()
        # and with the caller's permission to snapshot the values: the plan re-lays the matrix out as ELL
        plan3 = sp.CsrPlan(A.ptr, snapshot_values=True)
        r = bench_kernel(torch, sp, stream, lambda: plan3.spmv(x, y, s_ptr), csr_bytes, args.steps, args.warmup, dist_on, world)
        keep_output("config2_csr_planned_value_snapshot_y", y)
        extra["config2_csr_planned_value_snapshot"] = {
            "gbs": r4(r["gbs"]), "ms": r4(r["ms_per_step"]), "frac": r4(r["gbs"] / world / peak), "plan_mode": plan3.info()[2],
            "note": "CSR algorithmic bytes over the time of the ELL kernel the plan routes to (it moves 805 MB)"}
        plan3.close()
    sp.ell_destroy(E)
    del A, rp, ci, va, x, y, x_host, y_host, y_device_path
    torch.cuda.empty_cache()

    if not args.quick and not args.only_pagerank and world == 1:
        # ---- config 3: short rows + 4 outlier rows of 1 M nnz: scalar (reference policy) vs merge ---
        log("config 3")
        rows3 = args.c3_rows
        rp3, ci3, va3 = gen.short_rows_with_outliers_csr(rows3, 43, dev)
        A3 = sp.DeviceCSR(rows3, rows3, rp3, ci3, va3)
        x3 = gen.uniform_01_open_low(5, torch.arange(rows3, device=dev), 9)
        y3 = torch.empty(rows3, dtype=torch.float32, device=dev)
        b3 = sp.csr_bytes(rows3, rows3, ci3.numel())
        for kernel, name in ((sp.SCALAR_CSR, "csr_scalar"), (sp.MERGE_PATH, "csr_merge")):
            cfg = sp.make_config(kernel)
            r = bench_kernel(torch, sp, stream, lambda: sp.lib.spmv_b200_spmv_csr_async(
                A3.ptr, sp.dptr(x3), sp.dptr(y3), C.byref(cfg), C.c_void_p(s_ptr)), b3, args.steps, 3)
            extra[f"config3_{name}"] = {"gbs": r4(r["gbs"]), "ms": r4(r["ms_per_step"]), "frac": r4(r["gbs"] / peak),
                                        "rows": rows3, "nnz": ci3.numel()}
            keep_output(f"config3_{name}_y", y3)
        extra["config3_selector"] = "MERGE_PATH (outlier override; reference policy: SCALAR_CSR)"
        scalars["config3_merge_frac"] = extra["config3_csr_merge"]["frac"]
        del A3, rp3, ci3, va3, x3, y3
        torch.cuda.empty_cache()

    # ---- config 4: R-MAT SpMV through MERGE_PATH, row-sharded over the ranks (strong scaling) ------------
    def rmat_spmv_section(scale, seed):
        log(f"R-MAT scale {scale}: build")
        n, bounds, srp, sci, sva, n_edges = gen.rmat_pagerank_shard(scale, 16, seed, rank, world, dev, row_weight=1)
        torch.cuda.synchronize()
        rows_p = bounds[rank + 1] - bounds[rank]
        csr = sp.DeviceCSR(rows_p, n, srp, sci, sva)
        xg = torch.full((n,), 1.0 / n, dtype=torch.float32, device=dev)
        y_slice = torch.empty(max(rows_p, 1), dtype=torch.float32, device=dev)
        b4 = 8 * sci.numel() + 4 * (rows_p + 1) + 4 * n + 4 * rows_p
        tot4 = torch.tensor([float(b4)], dtype=torch.float64, device=dev)
        if dist_on:
            dist.all_reduce(tot4)
        tot = float(tot4.item())
        cfg = sp.make_config(sp.MERGE_PATH)
        log(f"R-MAT scale {scale}: csr_merge")
        r = bench_kernel(torch, sp, stream, lambda: sp.lib.spmv_b200_spmv_csr_async(
            csr.ptr, sp.dptr(xg), sp.dptr(y_slice), C.byref(cfg), C.c_void_p(s_ptr)), 0, args.steps, 3, dist_on)
        gbs = tot / (r["ms_per_step"] * 1e-3) / 1e9
        extra[f"rmat{scale}_csr_merge"] = {"gbs": r4(gbs), "ms": r4(r["ms_per_step"]), "frac": r4(gbs / world / peak),
                                           "nnz": n_edges, "rows": n, "scaling": "strong (one graph, row shards)"}
        torch.cuda.synchronize()
        y_ref = y_slice.clone()
        keep_output(f"rmat{scale}_csr_merge_y", y_ref[:rows_p])
        # the same product through a CSR plan: merge coordinates computed once + hub-column table
        # (csr_hot_kernels.cu) for scale-free shards; bit-identical results, checked here on the full-size shard
        log(f"R-MAT scale {scale}: csr_merge through a CSR plan")
        t0 = time.perf_counter()
        plan = sp.CsrPlan(csr.ptr)
        torch.cuda.synchronize()
        plan_ms = (time.perf_counter() - t0) * 1e3
        hot_columns, hot_nnz, hot_mode = plan.info()
        r = bench_kernel(torch, sp, stream, lambda: plan.spmv(xg, y_slice, s_ptr), 0, args.steps, 3, dist_on)
        torch.cuda.synchronize()
        keep_output(f"rmat{scale}_csr_merge_plan_y", y_slice[:rows_p])
        same = all_ok(bool(torch.equal(y_ref.view(torch.int32), y_slice.view(torch.int32))))
        gbs = tot / (r["ms_per_step"] * 1e-3) / 1e9
        extra[f"rmat{scale}_csr_merge_plan"] = {
            "gbs": r4(gbs), "ms": r4(r["ms_per_step"]), "frac": r4(gbs / world / peak), "hub_columns_rank0": hot_columns,
            "hub_nnz_fraction_rank0": r4(hot_nnz / max(sci.numel(), 1)), "plan_mode": hot_mode, "plan_build_ms": r4(plan_ms),
            "bit_identical_to_csr_merge": same}
        parity[f"rmat{scale}_plan_bit_identical_to_merge"] = same
        scalars[f"rmat{scale}_merge_ms"] = r4(r["ms_per_step"])
        scalars[f"rmat{scale}_merge_gbs"] = r4(gbs)
        scalars[f"rmat{scale}_merge_frac"] = r4(gbs / world / peak)
        plan.close()
        del csr, srp, sci, sva, xg, y_slice, y_ref
        torch.cuda.empty_cache()

    # ---- config 5: PageRank through the native sharded path (spmv_b200_pr_dist_*) ------------------------
    names = {"multicast": D.EXCHANGE_MULTICAST, "p2p": D.EXCHANGE_P2P, "nccl": D.EXCHANGE_NCCL}

    def pagerank_parity_small(scale=20, seed=45, iters=10):
        """Every transport on a scale-20 graph against the f64-accumulator restatement of the reference
        recurrence (oracle/, checker use only) at equal iteration count: L1 <= 1e-6, transports bit-identical."""
        log(f"parity: sharded PageRank at scale {scale} against the oracle")
        n, bounds, srp, sci, sva, _ = gen.rmat_pagerank_shard(scale, 16, seed, rank, world, dev, row_weight=4)
        torch.cuda.synchronize()
        csr = sp.DeviceCSR(bounds[rank + 1] - bounds[rank], n, srp, sci, sva)
        c = comm if dist_on else D.NativeComm(0, 1, session + "-p")
        vectors, used = {}, {}
        for name in (["multicast", "p2p", "nccl"] if dist_on else ["p2p"]):
            pr = D.NativeShardedPageRank(c, csr, bounds[rank], n, names[name])
            pr.run(0.85, 0.0, 0, fixed_iterations=iters)
            vectors[name] = pr.ranks(dev).clone()
            used[name] = D.EXCHANGE_NAMES[pr.exchange]
            pr.close()
        if not dist_on:
            c.close()
        keys = list(vectors)
        identical = all_ok(all(torch.equal(vectors[keys[0]].view(torch.int32), vectors[k].view(torch.int32)) for k in keys[1:]))
        l1 = -1.0
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from oracle_binding import Oracle
            orc = Oracle()
            _, frp, fci, fva = gen.rmat_pagerank_csr(scale, 16, seed, "cpu")
            o_ranks = orc.pagerank_f64(n, n, frp.numpy(), fci.numpy(), fva.numpy(), 0.85, 1e-6, 100, fixed_it=iters)[0]
            l1 = max(float(np.abs(vectors[k].cpu().numpy().astype(np.float64) - o_ranks).sum()) for k in keys)
        ok = all_ok(identical and (rank != 0 or l1 <= 1e-6))
        parity["pagerank_scale20"] = {"l1_vs_oracle_f64_max_over_transports": l1, "tolerance": 1e-6, "iterations": iters,
                                      "transports": used, "transports_bit_identical": identical, "ok": ok}
        return ok

    def pagerank_section(scale, seed, relabelled=False):
        tag = "_relabelled" if relabelled else ""
        graph_name = f"R-MAT scale {scale} x16, d=0.85" + (", vertex ids relabelled (Graph500-style)" if relabelled
                                                          else ", no vertex permutation")
        # a PageRank shard also updates and sends every owned row, so rows weigh more than in plain SpMV: the
        # local step costs nnz + 2.25 per row (scripts/shard_balance.py); with the 8-way exchange 4 measured best
        # (w = 1 / 2 / 4 / 8 -> 995 / 1132 / 1154 / 920 iter/s)
        weight = args.row_weight if args.row_weight >= 0 else (1 if world == 1 or relabelled else (2 if world == 2 else 4))
        log(f"PageRank {graph_name}: build shard (work(row) = nnz + {weight})")
        n, bounds, srp, sci, sva, n_edges = gen.rmat_pagerank_shard(scale, 16, seed, rank, world, dev, row_weight=weight,
                                                                    relabelled=relabelled)
        torch.cuda.synchronize()
        rows_p = bounds[rank + 1] - bounds[rank]
        csr = sp.DeviceCSR(rows_p, n, srp, sci, sva)
        it_bytes = 8 * sci.numel() + 4 * (rows_p + 1) + 4 * n + 4 * rows_p
        tot = torch.tensor([float(it_bytes)], dtype=torch.float64, device=dev)
        if dist_on:
            dist.all_reduce(tot)
        it_bytes = float(tot.item())
        c = comm if dist_on else D.NativeComm(0, 1, session + "-s" + tag)
        modes = ["p2p"] if not dist_on else (["multicast"] if relabelled else ["nccl", "p2p", "multicast"])
        iters = args.pr_iters
        best = None
        checks = {}
        for mode in modes:
            log(f"PageRank {graph_name}: {mode}")
            pr = D.NativeShardedPageRank(c, csr, bounds[rank], n, names[mode])
            used = D.EXCHANGE_NAMES[pr.exchange] if dist_on else "none (1 GPU)"
            sec = None
            link0 = None
            for rep in range(2):  # the first run also builds the dangling set and captures the CUDA graphs
                if rep == 1 and dist_on:
                    link0 = nvlink_bytes(local_rank)
                res = pr.run(0.85, 0.0, 0, fixed_iterations=iters)
                t = max_over_ranks(res.device_seconds)
                sec = t if sec is None else min(sec, t)
            link1 = nvlink_bytes(local_rank) if link0 is not None else None
            vec = pr.ranks(dev)
            if mode == modes[0]:  # the transports are checked bit-identical below
                keep_output(f"pagerank{tag}_ranks", vec)
            total = float(vec.double().sum().item())
            checks[mode] = vector_checksum(torch, vec) + (total,)
            entry = {"iters_per_s": r4(iters / sec), "ms_per_iter": r4(sec / iters * 1e3), "exchange": used,
                     "graph": graph_name, "n": n, "nnz": n_edges, "iterations_timed": iters,
                     "l2_residual_after": res.final_residual, "effective_gbs": r4(it_bytes / (sec / iters) / 1e9),
                     "frac": r4(it_bytes / (sec / iters) / 1e9 / world / peak), "cuda_graph_replay": bool(res.graph_replay),
                     "kernels_per_iteration": res.kernels_per_iteration, "hub_columns_rank0": pr.hub_columns,
                     "partition": f"work(row) = nnz + {weight}",
                     "rows_per_rank_max": int(max(bounds[i + 1] - bounds[i] for i in range(world))),
                     "timing": "CUDA events around the whole loop on every rank (inside spmv_b200_pr_dist_run), max over ranks; "
                               "excluded: set-up and the final normalisation"}
            if dist_on:
                # NVLink data counters of this rank's GPU around the timed run (driver counters, not a profiler):
                # egress / ingress per iteration, max over ranks -- the evidence for "multicast sends every row once"
                have = link0 is not None and link1 is not None
                tx = max_over_ranks((link1[0] - link0[0]) / res.iterations_launched if have else -1.0)
                rx = max_over_ranks((link1[1] - link0[1]) / res.iterations_launched if have else -1.0)
                entry["nvlink_tx_mb_per_iter_max_rank"] = r4(tx / 1e6) if tx >= 0 else None
                entry["nvlink_rx_mb_per_iter_max_rank"] = r4(rx / 1e6) if rx >= 0 else None
                entry["slice_bytes_max_rank"] = int(max(bounds[i + 1] - bounds[i] for i in range(world))) * 4
            extra[f"pagerank{tag}_{mode}" if dist_on else f"pagerank{tag}"] = entry
            if best is None or entry["iters_per_s"] > best[1]["iters_per_s"]:
                best = (mode, entry)
            pr.close()
        if not dist_on:
            c.close()
        # full-size parity: every rank holds the bit-identical vector, whatever the transport, and it sums to 1
        mine = torch.tensor([v for m in modes for v in checks[m][:2]], dtype=torch.int64, device=dev)
        ok = True
        if dist_on:
            gathered = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(gathered, mine)
            ok = all(bool(torch.equal(g, gathered[0])) for g in gathered)
        first = checks[modes[0]]
        same_transports = all(checks[m][:2] == first[:2] for m in modes)
        sum_ok = abs(first[2] - 1.0) <= 1e-6
        ok = all_ok(ok and same_transports and sum_ok)
        parity[f"pagerank_scale{scale}{tag}"] = {"ranks_bit_equal_across_gpus": ok if dist_on else None,
                                                  "transports_bit_identical": same_transports, "sum_of_ranks": first[2],
                                                  "ok": ok}
        del csr, srp, sci, sva
        torch.cuda.empty_cache()
        return best

    def pagerank_one_gpu(scale, seed):
        """The same graph, whole, on rank 0's GPU alone (the other ranks wait): the denominator of the
        1 -> N scaling figure, measured in the same run on the same box."""
        sec = 0.0
        if rank == 0:
            log(f"PageRank R-MAT {scale} on ONE GPU (scaling denominator)")
            n, bounds, srp, sci, sva, _ = gen.rmat_pagerank_shard(scale, 16, seed, 0, 1, dev, row_weight=1)
            torch.cuda.synchronize()
            csr = sp.DeviceCSR(n, n, srp, sci, sva)
            c1 = D.NativeComm(0, 1, session + "-one")
            pr = D.NativeShardedPageRank(c1, csr, 0, n, D.EXCHANGE_P2P)
            for _ in range(2):
                res = pr.run(0.85, 0.0, 0, fixed_iterations=args.pr_iters)
                sec = res.device_seconds if sec == 0.0 else min(sec, res.device_seconds)
            keep_output("pagerank_1gpu_ranks", pr.ranks(dev))
            pr.close()
            c1.close()
            del csr, srp, sci, sva
            torch.cuda.empty_cache()
        if dist_on:
            dist.barrier()
        return max_over_ranks(sec)

    parity_ok = True
    if not args.quick:
        if not args.only_pagerank:
            rmat_spmv_section(args.rmat_scale, 44)
        parity_ok = pagerank_parity_small() and parity_ok
        best = pagerank_section(args.pr_scale, 45)
        scalars["pagerank_iters_per_s"] = best[1]["iters_per_s"]
        scalars["pagerank_ms_per_iter"] = best[1]["ms_per_iter"]
        scalars["pagerank_exchange"] = best[0] if dist_on else "none (1 GPU)"
        scalars["pagerank_frac"] = best[1]["frac"]
        if dist_on:
            for mode in ("nccl", "p2p", "multicast"):
                e = extra.get(f"pagerank_{mode}")
                if e:
                    scalars[f"pagerank_{mode}_iters_per_s"] = e["iters_per_s"]
            if args.pr_one_gpu:
                one = pagerank_one_gpu(args.pr_scale, 45)
                scalars["pagerank_1gpu_iters_per_s"] = r4(args.pr_iters / one)
                scalars["pagerank_1gpu_ms_per_iter"] = r4(one / args.pr_iters * 1e3)
                scalars["pagerank_speedup_vs_1gpu"] = r4(best[1]["iters_per_s"] / (args.pr_iters / one))
        else:
            scalars["pagerank_1gpu_iters_per_s"] = best[1]["iters_per_s"]
        if args.relabelled:
            best_r = pagerank_section(args.pr_scale, 45, relabelled=True)
            scalars["pagerank_relabelled_iters_per_s"] = best_r[1]["iters_per_s"]
    parity_ok = parity_ok and all(v.get("ok", True) if isinstance(v, dict) else bool(v) for v in parity.values())
    parity["ok"] = parity_ok

    if rank == 0:
        traffic, traffic_src = ncu_traffic_for("ell_tma_pipe_kernel<1>") if world == 1 else (None, "N > 1: not captured")
        if args.ncu_traffic is not None:
            traffic, traffic_src = args.ncu_traffic, "--ncu-traffic"
        roofline = {"bound": "hbm", "achieved": launch_gbs, "peak": peak, "unit": "GB/s", "frac": launch_gbs / peak,
                    "peak_source": peak_src, "frac_of_8000_nominal": launch_gbs / 8000.0,
                    "kernel": "ell_tma_pipe_kernel<1>", "algorithmic_bytes_per_launch": ell_bytes,
                    "traffic": traffic, "traffic_source": traffic_src}
        config = headline_config(n_loc * world, nnz_total, ell_bytes * world, world)
        config.update(scalars)
        line = {
            "metric": "spmv_effective_hbm_gbs", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity": parity,
        }
        line.update(scalars)
        line["extra"] = extra
        if args.dump_outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if comm is not None:
        comm.close()
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()
    if not parity_ok:
        raise SystemExit("bench.py: PARITY FAILURE -- " + json.dumps(parity))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--quick", action="store_true", help="headline + e2e + cpu baseline only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rmat-scale", type=int, default=24, help="BASELINE config 4: R-MAT SpMV")
    ap.add_argument("--pr-scale", type=int, default=26, help="BASELINE config 5: PageRank graph")
    ap.add_argument("--c3-rows", type=int, default=50_000_000)
    ap.add_argument("--pr-iters", type=int, default=20)
    ap.add_argument("--row-weight", type=int, default=-1, help="partition work(row) = nnz + row_weight (-1: default policy)")
    ap.add_argument("--only-pagerank", action="store_true", help="tuning aid: headline + PageRank section only")
    ap.add_argument("--relabelled", type=int, default=1,
                    help="also run PageRank on the same R-MAT graph with relabelled vertex ids (extra.pagerank_relabelled)")
    ap.add_argument("--ncu-traffic", type=float, default=None,
                    help="dram bytes per launch of the dominant kernel from an ncu capture (default: profiles/ncu_traffic.json, "
                         "N = 1 only)")
    ap.add_argument("--pr-one-gpu", type=int, default=1,
                    help="N > 1: rank 0 also runs the whole PageRank graph on its GPU alone (pagerank_1gpu_iters_per_s, "
                         "pagerank_speedup_vs_1gpu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed seeded sample of every timed path's output after its last step as DIR/<name>.npy "
                         "(float32, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_product_arm(args)


if __name__ == "__main__":
    main()
