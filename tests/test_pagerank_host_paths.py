"""Single-GPU PageRank through each host path, with and without CUDA-graph replay of the iterations.

pagerank_device runs the one-kernel loop on small graphs and the multi-kernel loop elsewhere; the multi-kernel loop
steps with the plain merge tile, the segmented stream or the hub-column kernel, and replays its two ping-pong
iterations from CUDA graphs unless SPMV_B200_PR_GRAPH=0.  The variables are read once per process, so each
(path, graph) pair runs in a child process (this file with --child) and prints a fingerprint: ranks (sha256 of the
bits), iterations, residual, L2 history and the launch_count() delta of pagerank_device_history; the same for a
personalized run, pagerank() and the sharded loop at world 1.  Graph replay and the eager loop must agree bit for bit
with the same launch count.  The FINGERPRINT lines (pytest -s) let two builds be compared path by path."""
import functools
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V = "SPMV_B200_"
# path -> (variables, R-MAT (scale, edge factor, seed))
PATHS = {
    "small": ({}, (10, 8, 3)),
    "tile": ({V + "HOT": "0", V + "PR_SMALL": "0"}, (12, 8, 5)),
    "seg": ({V + "PLAN": "seg", V + "HOT": "1", V + "PR_SMALL": "0"}, (12, 8, 6)),
    "hub_all_x": ({V + "PLAN": "hub", V + "HOT": "1", V + "PR_SMALL": "0"}, (12, 8, 7)),
    "hub_table": ({V + "PLAN": "hub", V + "HOT": "1", V + "PR_SMALL": "0"}, (17, 4, 8)),
}
CONFIGS = {"converging": (0.85, 1e-6, 100), "fixed_6": (0.85, 0.0, 6)}  # 6: still graph-captured (>= 4)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _sha(a):
    return hashlib.sha256(_bits(a).tobytes()).hexdigest()[:16]


def _f32hex(x):
    return "%08x" % int(_bits(np.float32(x)).reshape(-1)[0])


def child_main(path):
    import torch
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    from _load_pkg import load_pkg
    sp = load_pkg()
    import gpu_spmv_b200.dist as Dm
    import gpu_spmv_b200.gen as gen
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    scale, ef, seed = PATHS[path][1]
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, ef, seed, "cpu")
    G = sp.DeviceCSR(n, n, rp.to(dev), ci.to(dev), va.to(dev))
    out = {}
    for name, (d, tol, it) in CONFIGS.items():
        d_ranks = torch.full((n,), float("nan"), dtype=torch.float32, device=dev)
        before = sp.launch_count()
        rc, iters, res, conv, hist = sp.pagerank_device_history(G.ptr, d_ranks, sp.make_pagerank_config(d, tol, it), 128)
        torch.cuda.synchronize()
        out[name] = {"rc": rc, "iterations": iters, "residual": _f32hex(res), "converged": bool(conv),
                     "history": _sha(hist[:iters]), "ranks": _sha(d_ranks.cpu().numpy()),
                     "launches": sp.launch_count() - before}
    v = np.random.default_rng(seed).uniform(0, 1, n).astype(np.float32)
    v[v < 0.9] = 0
    d_ranks = torch.empty(n, dtype=torch.float32, device=dev)
    before = sp.launch_count()
    rc, iters, res, conv, l1, hist = sp.pagerank_device_personalized(G.ptr, d_ranks, v, sp.make_pagerank_config(), 128)
    out["personalized"] = {"rc": rc, "iterations": iters, "residual": _f32hex(res), "l1": float(l1).hex(),
                           "history": _sha(hist[:iters]), "ranks": _sha(d_ranks.cpu().numpy()),
                           "launches": sp.launch_count() - before}
    A = sp.csr_from_arrays(n, n, rp.numpy(), ci.numpy(), va.numpy())
    assert sp.csr_to_gpu(A) == 0
    result, ranks = sp.pagerank(A, sp.make_pagerank_config())
    out["pagerank"] = {"iterations": result.iterations, "residual": _f32hex(result.final_residual),
                       "converged": bool(result.converged), "ranks": _sha(ranks)}
    sp.pagerank_free(result)
    sp.csr_destroy(A)
    comm = Dm.NativeComm(0, 1, f"hostpaths-{path}-{os.getpid()}")
    pr = Dm.NativeShardedPageRank(comm, G, 0, n, Dm.EXCHANGE_P2P)
    try:
        runs = []
        for _ in range(2):  # the second run replays the graphs the first one captured
            res = pr.run(0.85, 1e-6, 100)
            runs.append({"iterations": res.iterations, "launched": res.iterations_launched,
                         "residual": _f32hex(res.final_residual), "graph_replay": res.graph_replay,
                         "kernels_per_iteration": res.kernels_per_iteration, "ranks": _sha(pr.ranks(dev).cpu().numpy())})
        out["dist"] = {"runs": runs, "hub_columns": pr.hub_columns}
    finally:
        pr.close()
        comm.close()
    print("RESULT " + json.dumps(out), flush=True)


@functools.lru_cache(maxsize=None)
def run_child(path, graph):
    env = {k: v for k, v in os.environ.items() if not k.startswith(V)}
    env.update(PATHS[path][0])
    if not graph:
        env[V + "PR_GRAPH"] = "0"
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    recs = [json.loads(line[7:]) for line in p.stdout.splitlines() if line.startswith("RESULT ")]
    assert p.returncode == 0 and len(recs) == 1, p.stdout[-4000:]
    print(f"FINGERPRINT {path} graph={int(graph)} {json.dumps(recs[0], sort_keys=True)}")
    return recs[0]


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_graph_replay_matches_eager_loop(cuda, path):
    g, e = run_child(path, True), run_child(path, False)
    for name in list(CONFIGS) + ["personalized"]:
        assert g[name]["rc"] == 0 and g[name]["iterations"] > 0, (name, g[name])
        assert g[name] == e[name], f"{name}: graph replay {g[name]} != eager loop {e[name]}"
    assert g["pagerank"] == e["pagerank"]
    assert g["converging"]["converged"] and g["converging"]["iterations"] > 6
    assert not g["fixed_6"]["converged"] and g["fixed_6"]["iterations"] == 6
    # the one-kernel loop launches the same kernels however many iterations it runs; the multi-kernel loop does not
    small = g["converging"]["launches"] == g["fixed_6"]["launches"]
    assert small == (path == "small"), (g["converging"], g["fixed_6"])
    if path == "tile":
        assert g["dist"]["hub_columns"] == 0
    if path.startswith("hub"):
        assert g["dist"]["hub_columns"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_sharded_world_one_replays_graphs(cuda, path):
    g, e = run_child(path, True), run_child(path, False)
    for runs, replay in ((g["dist"]["runs"], 1), (e["dist"]["runs"], 0)):
        assert [r["graph_replay"] for r in runs] == [replay, replay], runs
        assert runs[0] == runs[1], runs
    kpi = g["dist"]["runs"][0]["kernels_per_iteration"]
    assert kpi > 0 and e["dist"]["runs"][0]["kernels_per_iteration"] == 0
    strip = lambda r: {k: v for k, v in r.items() if k not in ("graph_replay", "kernels_per_iteration")}  # noqa: E731
    assert strip(g["dist"]["runs"][0]) == strip(e["dist"]["runs"][0])


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    child_main(sys.argv[2])
