"""Runs the sharded PageRank loop (one rank) several times on one GPU and checks bitwise reproducibility."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from _load_pkg import load_pkg
sp = load_pkg()
import gpu_spmv_b200.dist as D
import gpu_spmv_b200.gen as gen
dev = torch.device("cuda:0")
torch.cuda.set_device(0)
scale = int(sys.argv[1]) if len(sys.argv) > 1 else 22
n, rp, ci, va = gen.rmat_pagerank_csr(scale, 16, 44, dev)
G = sp.DeviceCSR(n, n, rp, ci, va)
torch.cuda.synchronize()
comm = D.NativeComm(0, 1, f"check-determinism-{os.getpid()}")
pr = D.NativeShardedPageRank(comm, G, 0, n)
outs = []
try:
    for rep in range(4):
        res = pr.run(0.85, 0.0, 24, fixed_iterations=24)
        outs.append(pr.ranks(dev).clone())
        print(rep, "iters", res.iterations, "residual", res.final_residual, "l1", res.l1_residual,
              "exchange", D.EXCHANGE_NAMES.get(res.exchange), "graph replay", res.graph_replay, flush=True)
finally:
    pr.close()
    comm.close()
for o in outs[1:]:
    print("bitwise equal to run 0:", bool(torch.equal(o.view(torch.int32), outs[0].view(torch.int32))))
