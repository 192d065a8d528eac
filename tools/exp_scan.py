"""Scan-kernel experiment driver: build an index of a given shape on the GPU, then time the batched scan for a
list of (variant, streams) settings.  Used for A/B runs and as the ncu target for the scan kernels.
usage: python tools/exp_scan.py --rows 1000000 --dim 128 --ef 40 [--opclass vector_l2_ops] [--variants 0,6,9]
                                [--streams 1,3] [--steps 10] [--nq 10000] [--latency]"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import pgvector_hnsw_partitioning_b200 as pkg  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1000000)
ap.add_argument("--dim", type=int, default=128)
ap.add_argument("--ef", type=int, default=40)
ap.add_argument("--nq", type=int, default=10000)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--opclass", default="")
ap.add_argument("--variants", default="0")
ap.add_argument("--streams", default="1,3")
ap.add_argument("--latency", action="store_true", help="also time single scans through hb_rescan + hb_gettuple")
ap.add_argument("--latency-variants", default="", help="variants to repeat the latency loop under (6 = no CTA-per-query kernel)")
ap.add_argument("--seed", type=int, default=20260103)
ap.add_argument("--slots", type=int, default=0, help="visited-table slots (0 = automatic)")
a = ap.parse_args()

dev = torch.device("cuda", 0)
opc = a.opclass or ("vector_l2_ops" if a.dim == 128 else "vector_cosine_ops")
half = opc.startswith("halfvec")
x = bench.gen_set(a.rows, a.dim, a.seed, dev)
xs = x.half() if half else x
xh = xs.cpu().numpy()
ix, n, dt = bench.build_index(pkg, xh, a.dim, 0, opclass=opc)
print("build %.2fs (%.0f vectors/s)" % (dt, n / dt), flush=True)
ix.trim()
row = a.dim * (2 if half else 4)
nsteps = a.steps
q_all = bench.gen_set(a.nq * (nsteps + 3), a.dim, a.seed + 1000, dev)
if half:
    q_all = q_all.half()
q_all = q_all.view(nsteps + 3, a.nq, a.dim)
metric = "l2" if "_l2_" in opc else ("ip" if "_ip_" in opc else "cosine")
gt = bench.exact_topk_metric(xs, q_all[0][:1000], 10, metric)
del x, xs
if a.slots:
    ix.set_option("slots", a.slots)
for variant in [int(v) for v in a.variants.split(",")]:
    ix.set_option("variant", variant)
    for ns in [int(s) for s in a.streams.split(",")]:
        streams = [torch.cuda.Stream(device=dev) for _ in range(ns)]
        outs = [(torch.empty((a.nq, a.ef), dtype=torch.int32, device=dev), torch.empty((a.nq, a.ef), dtype=torch.float32, device=dev),
                 torch.empty((a.nq,), dtype=torch.int32, device=dev)) for _ in range(ns)]
        main = torch.cuda.current_stream(dev)

        def run(first, count):
            for st in streams:
                st.wait_stream(main)
            for s in range(count):
                st, (e_, d_, c_) = streams[s % ns], outs[s % ns]
                ix.search_dev(q_all[first + s].data_ptr(), a.nq, a.ef, e_.data_ptr(), d_.data_ptr(), c_.data_ptr(), st.cuda_stream)
            for st in streams:
                main.wait_stream(st)

        run(0, 3)
        run(0, 3)
        torch.cuda.synchronize()
        ix.search_dev(q_all[0].data_ptr(), a.nq, a.ef, outs[0][0].data_ptr(), outs[0][1].data_ptr(), outs[0][2].data_ptr(), streams[0].cuda_stream)
        torch.cuda.synchronize()
        rec = bench.recall_at(outs[0][0][:1000, :10].cpu().numpy(), gt)
        ix.counters(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        run(3, nsteps)
        e1.record(main)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / nsteps
        c = ix.counters(reset=True)
        alg = (c["n_dist"] * row + c["n_hop0"] * 128 + c["n_hopu"] * 64 + a.nq * nsteps * row) / nsteps
        print("variant=%d streams=%d: %.3f ms/step  %.0f QPS  %.0f GB/s alg (%.3f of 6456)  n_dist/q=%.1f hops/q=%.1f slow=%d recall@10=%.4f"
              % (variant, ns, ms, a.nq / ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 6455.9, c["n_dist"] / a.nq / nsteps,
                 (c["n_hop0"] + c["n_hopu"]) / a.nq / nsteps, c["n_slow"], rec), flush=True)
for lv in ([int(v) for v in a.latency_variants.split(",")] if a.latency_variants else [None]) if a.latency else []:
    if lv is not None:
        ix.set_option("variant", lv)
        print("latency under variant %d" % lv, flush=True)
    qh = q_all[1][:200].cpu().numpy()
    sc = ix.beginscan()
    for i in range(20):
        sc.rescan(qh[i], a.ef)
        sc.gettuple()
    t0 = time.perf_counter()
    for i in range(20, 200):
        sc.rescan(qh[i], a.ef)
        sc.gettuple()
    dt = (time.perf_counter() - t0) / 180
    sc.endscan()
    print("hb_rescan + first hb_gettuple: %.1f us" % (dt * 1e6), flush=True)
    for nqs in (1, 8, 32, 64, 148, 512):
        qs = qh[:nqs] if nqs <= 200 else np.tile(qh, (3, 1))[:nqs]
        for r in range(3):
            ix.search(qs, 10, a.ef)
        t0 = time.perf_counter()
        for r in range(20):
            ix.search(qs, 10, a.ef)
        print("hb_search_batch nq=%d: %.1f us" % (nqs, (time.perf_counter() - t0) / 20 * 1e6), flush=True)
