"""Time the exact scan (config 5) at the C2 shape.  usage: python tools/exp_bf.py [n] [nq]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import pgvector_hnsw_partitioning_b200 as pkg
from bench import gen_set, exact_topk_metric, recall_at

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
nq = int(sys.argv[2]) if len(sys.argv) > 2 else 10000
dim = 768
dev = torch.device("cuda", 0)
x = gen_set(n, dim, 20260102, dev)
ix = pkg.HnswIndex(dim, "vector_cosine_ops", 16, 64, capacity=n)
xn = torch.nn.functional.normalize(x, dim=1).cpu().numpy()
g = type("G", (), {})()
g.dim, g.m, g.efc, g.n, g.upper_rows, g.entry = dim, 16, 64, n, 0, 0
g.vecs, g.level, g.nbr0 = xn, np.zeros(n, np.uint8), np.full((n, 32), -1, np.int32)
g.uoff, g.nbru, g.ntids, g.tids = np.full(n, -1, np.int32), np.full((1, 16), -1, np.int32), np.ones(n, np.uint8), np.zeros((n, 10), np.int64)
ix.load_graph(g)
q = gen_set(nq, dim, 20260102 + 1000, dev)
qh = q.cpu().numpy()
for it in range(3):
    t0 = time.time()
    elem, dist, st = ix.bruteforce(qh, 10, stats=True)
    dt = time.time() - t0
    tf = 2.0 * nq * n * dim / (st["gemm_ms"] * 1e-3) / 1e12
    print("iter %d: total %.1f ms, gemm %.2f ms = %.0f TFLOP/s, certified %d rescanned %d, %.0f QPS (whole call)" %
          (it, dt * 1e3, st["gemm_ms"], tf, st["certified"], st["rescanned"], nq / dt), flush=True)
gt = exact_topk_metric(x, q[:1000], 10, "cosine")
print("agreement with torch fp32 top-10:", recall_at(elem[:1000], gt))
