#!/usr/bin/env python
"""bench.py -- headline benchmark of the HNSW hot path on B200.

Metric (BASELINE.json): QPS at recall@10 >= 0.95 on 1M x 768 fp32 cosine (configs[1]); also reports
HNSW build vectors/s and, at every N, the hash-partitioned search (configs[2]) and build (configs[3]).
One "step" = one pass of the batched scan (hnswgettuple for nq queries) over one batch of synthetic queries.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...        (one rank per GPU)

The one JSON line:
  value / roofline / e2e   configs[1].  N = 1: the single 1M x 768 index.  N > 1: a single unpartitioned graph
                           does not shard (SURVEY.md 8e), so every rank holds a replica and scans its own
                           query batches: "replicas only", weak scaling, no data-path collective.
  partitioned              configs[2]: 10M x 128 L2 in 8 hash partitions spread over the N ranks (hb_part_*:
                           scans -> device merge -> one ncclAllGather -> merge, three batches in flight);
                           strong scaling (same 10 000-query batches at every N).
  build_partitioned        configs[3]: 1M x 1536 halfvec inner-product index build, 8 partitions over the N ranks.
  cpu_baseline, parity     N = 1 only: the oracle (CPU restatement of pgvector's HNSW path) timed on the host cores
                           in a CHILD PROCESS that maps neither CUDA nor the product library, on the graph the GPU
                           built; its ids for the same queries are compared with the GPU's.
`--workload partitioned|build` print a line for those shapes alone.

`--dump-outputs DIR` (configs[1]): after the timed steps, rank 0 writes what the last timed step's scan returned
as DIR/elements.npy (element ids, -1 past the count), DIR/distances.npy (+inf past the count) and DIR/counts.npy,
one row per query, plus DIR/rows.npy (the query rows written).  Ids and counts are stored as float64, which holds
them exactly; distances as float32.  Above 64 MB in all, a fixed seeded sample of the queries is written.  Inputs
depend on the arguments only, so two builds of the project can be compared output for output.

`--impl reference`: the reference's CPU path.  The mount has no source and there is no PostgreSQL
(/root/reference/README.md:1), so what is timed is the C oracle (oracle/, "CPU restatement of pgvector HNSW
semantics -- not pgvector") with pgvector's natural summation order, on all host threads, over a bounded
sample of the same workload, in the same child process as `cpu_baseline` uses.  The parent builds the
1M-element graph on the GPU in untimed set-up (a single-threaded CPU build of 1M x 768 takes ~20 min) and hands
the flat image over through /dev/shm.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
FALLBACK_BF16_TFLOPS = 1400.0
NSLOT = 3                   # batches in flight (streams / async slots)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_JSON_FD = None


def own_stdout():
    """stdout must carry the one JSON line and nothing else, but native libraries write there too (NCCL prints its
    version banner at the first communicator): keep the real stdout aside for emit() and point fd 1 at stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), float(j.get("bf16_tflops", FALLBACK_BF16_TFLOPS)), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, FALLBACK_BF16_TFLOPS, "fallback"


def measured_traffic(kind, **key):
    """DRAM bytes per launch from the round's ncu captures (profiles/traffic.json, written by
    profiles/summarize.py --traffic); None when no capture matches this exact workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            for rec in json.load(f):
                if rec.get("kind") == kind and all(rec.get(k) == v for k, v in key.items()):
                    return rec
    except Exception:
        pass
    return None


def gen_set(n, dim, seed, device, n_centres=4096, latent=64, spread=0.35, noise=0.1, centre_seed=20260101):
    """SURVEY.md 8(d) C2 generator: mixture of Gaussian centres in a low-dimensional latent,
    random projection to `dim`, isotropic noise.  Not normalised (the cosine opclass does that)."""
    import torch
    gc = torch.Generator(device=device).manual_seed(centre_seed)
    cent = torch.randn((n_centres, latent), generator=gc, device=device)
    proj = torch.randn((latent, dim), generator=gc, device=device) / latent ** 0.5
    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty((n, dim), dtype=torch.float32, device=device)
    step = 1 << 18
    for s in range(0, n, step):
        e = min(n, s + step)
        a = torch.randint(0, n_centres, (e - s,), generator=g, device=device)
        z = cent[a] + spread * torch.randn((e - s, latent), generator=g, device=device)
        x = z @ proj
        x = x + noise * torch.randn((e - s, dim), generator=g, device=device)
        out[s:e] = x
    return out


def exact_topk_metric(x_dev, q_dev, k, metric):
    """torch fp32 exact top-k for l2 / ip / cosine (checker for recall only)."""
    import torch
    x = x_dev.float()
    q = q_dev.float()
    if metric == "cosine":
        x = torch.nn.functional.normalize(x, dim=1)
        q = torch.nn.functional.normalize(q, dim=1)
    xx = (x * x).sum(1) if metric == "l2" else None
    out = []
    for s in range(0, q.shape[0], 128):
        sims = q[s:s + 128] @ x.T
        if metric == "l2":
            sims = 2 * sims - xx[None, :]
        out.append(torch.topk(sims, k, dim=1).indices)
    return torch.cat(out).cpu().numpy()


def recall_at(ids, gt):
    return float(np.mean([len(set(ids[i]) & set(gt[i])) / gt.shape[1] for i in range(gt.shape[0])]))


DUMP_LIMIT = 64 * 10 ** 6


def dump_outputs(d, arrays, limit=DUMP_LIMIT):
    """Writes arrays that share a first axis (one row per query) as d/<name>.npy: integers as float64 (exact up to
    2**53), floats as float32.  When the files would exceed `limit` bytes, the same fixed seeded sample of rows is
    written from every array.  d/rows.npy lists the rows written."""
    arrays = {k: np.asarray(a, np.float64 if np.issubdtype(np.asarray(a).dtype, np.integer) else np.float32)
              for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_row = 8 + sum(a[:1].nbytes for a in arrays.values())
    budget = limit - 1024 * (len(arrays) + 1)          # .npy headers
    rows = np.arange(n)
    if n * per_row > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // per_row, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "rows.npy"), rows.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), a[rows])


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_index(pkg, x_host, dim, device_index, opclass="vector_cosine_ops", m=16, efc=64, seed=1):
    # warm-up: a 4096-row throwaway index loads the build kernels' modules (CUDA loads them lazily at first
    # launch) so that the timed build measures the build
    warm = pkg.HnswIndex(dim, opclass, m, efc, capacity=4096, device=device_index, seed=seed)
    warm.build(x_host[:4096])
    warm.close()
    ix = pkg.HnswIndex(dim, opclass, m, efc, capacity=x_host.shape[0], device=device_index, seed=seed)
    t0 = time.time()
    n = ix.build(x_host)
    dt = time.time() - t0
    return ix, n, dt


def pick_ef(ix, q_dev, gt, nq_eval, efs, stream, torch, target=0.95):
    sweep = []
    chosen = None
    for ef in efs:
        elem = torch.empty((nq_eval, ef), dtype=torch.int32, device=q_dev.device)
        dist = torch.empty((nq_eval, ef), dtype=torch.float32, device=q_dev.device)
        cnt = torch.empty((nq_eval,), dtype=torch.int32, device=q_dev.device)
        ix.search_dev(q_dev.data_ptr(), nq_eval, ef, elem.data_ptr(), dist.data_ptr(), cnt.data_ptr(), stream)
        torch.cuda.synchronize()
        r = recall_at(elem[:, :10].cpu().numpy(), gt)
        sweep.append({"ef_search": ef, "recall@10": round(r, 4)})
        if chosen is None and r >= target:
            chosen = (ef, r)
            break
    if chosen is None:
        chosen = (efs[-1], sweep[-1]["recall@10"])
    return chosen[0], chosen[1], sweep


# ---------------------------------------------------------------------------------------------------
# the CPU arm: oracle/cpu_arm.py in a child process (never imports torch, CUDA or the product package)
# ---------------------------------------------------------------------------------------------------
def shm_dir():
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return tempfile.mkdtemp(prefix="hb_bench_", dir=base)


def write_graph_image(ix, d):
    """The flat graph image (DESIGN.md 2) of a GPU-resident index as .npy files + meta.json."""
    g = ix.export_graph()
    for k in ("vecs", "level", "nbr0", "uoff", "nbru", "ntids", "tids"):
        np.save(os.path.join(d, k + ".npy"), getattr(g, k))
    json.dump({"dim": g.dim, "m": g.m, "efc": g.efc, "metric": g.metric, "dtype": g.dtype, "n": g.n, "upper_rows": g.upper_rows,
               "entry": g.entry[0] if isinstance(g.entry, tuple) else g.entry}, open(os.path.join(d, "meta.json"), "w"))


def run_cpu_child(job, d):
    jp = os.path.join(d, "job.json")
    json.dump(job, open(jp, "w"))
    env = dict(os.environ)
    env["CUDA_VISIBLE_DEVICES"] = ""          # the child has no business with the GPU
    p = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "cpu_arm.py"), jp], capture_output=True, text=True, env=env)
    if p.returncode != 0:
        raise RuntimeError("oracle/cpu_arm.py failed: " + p.stderr[-500:])
    return json.loads(p.stdout.strip().splitlines()[-1])


def cpu_search_arm(ix, q_eval_host, ef, steps, warmup, budget_s, parity, build_rows=None, build_meta=None):
    """Shared by `cpu_baseline` (ours arm) and `--impl reference`: same child, same method, same sample rule."""
    d = shm_dir()
    try:
        write_graph_image(ix, d)
        np.save(os.path.join(d, "queries.npy"), q_eval_host)
        job = {"graph_dir": d, "queries": os.path.join(d, "queries.npy"), "ef": ef, "steps": steps, "warmup": warmup,
               "budget_s": budget_s, "threads": 0, "parity": parity, "parity_out": os.path.join(d, "parity.npz")}
        if build_rows is not None:
            np.save(os.path.join(d, "rows.npy"), build_rows)
            job["build"] = dict(build_meta, rows=os.path.join(d, "rows.npy"))
        res = run_cpu_child(job, d)
        par = dict(np.load(os.path.join(d, "parity.npz"))) if parity else None
        return res, par
    finally:
        shutil.rmtree(d, ignore_errors=True)


def cpu_baseline_record(res, nq, ef):
    return {"value": round(res["queries_per_s"], 1), "unit": "queries/s", "cores": res["threads"], "kind": "port",
            "sample": "%d queries per step (bounded sample of the %d-query batch, same distribution), ef_search=%d, %d host "
                      "threads (one backend per thread), child process without CUDA; single thread: %.1f queries/s. CPU "
                      "restatement of pgvector HNSW semantics, not pgvector: no buffer manager/WAL, so faster than the real "
                      "extension" % (res["per_step"], nq, ef, res["threads"], res["single_thread_queries_per_s"]),
            "single_thread_value": round(res["single_thread_queries_per_s"], 1), "ms_per_step": round(res["ms_per_step"], 3)}


def parity_record(par, gpu_elem, gpu_dist, k=10):
    """GPU ids on the full-size graph vs the oracle's for the same queries: canonical order must be bit-identical;
    pgvector's natural order may differ only where distances tie within 1e-5 relative (north_star)."""
    n = par["canon_ids"].shape[0]
    ef = par["canon_ids"].shape[1]
    ce, cd = par["canon_ids"], par["canon_dist"]
    ne, nd = par["nat_ids"], par["nat_dist"]
    ids_identical = int(((gpu_elem[:n] == ce).all(axis=1)).sum())
    dist_identical = int(((gpu_dist[:n].view(np.uint32) == cd.view(np.uint32)).all(axis=1)).sum())
    kk = min(k, ef)
    nat_same, nat_tie, nat_bad = 0, 0, 0
    for i in range(n):
        if (ne[i, :kk] == gpu_elem[i, :kk]).all():
            nat_same += 1
            continue
        a, b = set(ne[i, :kk].tolist()), set(gpu_elem[i, :kk].tolist())
        dmap = dict(zip(gpu_elem[i].tolist(), gpu_dist[i].tolist()))
        dmap.update(dict(zip(ne[i].tolist(), nd[i].tolist())))
        edge = max(float(gpu_dist[i, kk - 1]), float(nd[i, kk - 1]))
        ok = all(abs(dmap[e] - edge) <= 1e-5 * max(abs(edge), 1e-3) for e in a ^ b)
        # same set in another order: neighbouring distances swapped within tolerance
        if ok and a == b:
            ok = bool(np.all(np.abs(np.asarray(nd[i, :kk]) - np.asarray(gpu_dist[i, :kk])) <= 1e-5 * np.maximum(np.abs(nd[i, :kk]), 1e-3)))
        if ok:
            nat_tie += 1
        else:
            nat_bad += 1
    return {"of": int(n), "ef_search": int(ef), "canonical_order": {"ids_identical": ids_identical, "distances_bit_identical": dist_identical},
            "natural_order_top%d" % kk: {"ids_identical": nat_same, "within_1e-5_ties": nat_tie, "unexplained": nat_bad},
            "note": "oracle = CPU restatement (parity unpinned against pgvector itself: the reference mount has no source)"}


WORKLOAD_C2 = "configs[1]: %dx%d fp32 cosine, m=16, ef_construction=64, ef_search=%d, k=10, %d queries/step"


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "partitioned", "build"])
    ap.add_argument("--rows", dest="n", type=int, default=0,
                    help="rows (0 = the configuration's own: 1M for configs[1], --part-rows for --workload partitioned, --build-rows for --workload build)")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", dest="nq", type=int, default=10000)
    ap.add_argument("--ef", type=int, default=0, help="hnsw.ef_search (0 = smallest of the sweep reaching recall 0.95)")
    ap.add_argument("--partitions", type=int, default=8)
    ap.add_argument("--part-rows", type=int, default=10000000, help="rows of the configs[2] sub-record")
    ap.add_argument("--build-rows", type=int, default=1000000, help="rows of the configs[3] sub-record")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work for the search baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the partitioned / build_partitioned sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's scan outputs as DIR/<name>.npy (configs[1], --impl ours)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs writes the configs[1] scan of --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference" and rank != 0:
        return 0
    own_stdout()
    # stdout carries the one JSON line and nothing else: NCCL's banner ("NCCL version ...") goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    import torch
    import pgvector_hnsw_partitioning_b200 as pkg

    if not torch.cuda.is_available():
        if args.impl == "reference":
            emit({"impl": "reference", "unavailable": "no CUDA device to build the 1M-element graph the CPU path searches"})
            return 0
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1 and args.impl == "ours":
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    rows_given = args.n > 0
    if not rows_given:
        args.n = 1000000
    n, dim, nq, k = args.n, args.dim, args.nq, 10
    hbm_peak, bf16_peak, peak_kind = peaks()
    ctx = dict(pkg=pkg, torch=torch, dev=dev, rank=rank, local_rank=local_rank, world=world, hbm_peak=hbm_peak, peak_kind=peak_kind)
    base_seed = 20260101 + 1
    if args.workload == "partitioned" and args.impl == "ours":
        rec = run_partitioned(args, ctx, args.n if rows_given else args.part_rows, args.dim if args.dim != 768 else 128)
        if rank == 0:
            emit(standalone_line(rec, world, args))
        return finish(torch, world)
    if args.workload == "build" and args.impl == "ours":
        rec = run_build_partitioned(args, ctx, args.n if rows_given else args.build_rows, args.dim if args.dim != 768 else 1536)
        if rank == 0:
            emit(standalone_line(rec, world, args))
        return finish(torch, world)

    # ---------------------------------------------------------------- data + index (untimed)
    t0 = time.time()
    x_dev = gen_set(n, dim, base_seed, dev)
    x_host = x_dev.cpu().numpy()
    log("[rank %d] generated %d x %d in %.1fs" % (rank, n, dim, time.time() - t0))
    ix, n_indexed, build_s = build_index(pkg, x_host, dim, local_rank)
    bc = ix.counters(reset=True)
    log("[rank %d] built %d elements in %.1fs (%.0f vectors/s)" % (rank, n_indexed, build_s, n_indexed / build_s))
    row_bytes = dim * 4

    # queries: a distinct batch per step, different for every rank
    total_steps = args.warmup + args.steps
    nq_eval = min(4000, nq)      # recall is estimated on 4000 queries: the 0.95 threshold is decided within ~0.2 pt
    q_eval = gen_set(nq_eval, dim, base_seed + 1000, dev)
    # ground truth: the library's exact scan (bf16 tcgen05 GEMM + fp32 re-rank, certified), cross-checked
    # against a plain torch fp32 scan
    gt_torch = exact_topk_metric(x_dev, q_eval, k, "cosine")
    del x_dev
    gt, _, bf_stats = ix.bruteforce(q_eval.cpu().numpy(), k, stats=True)
    gt_agree = recall_at(gt, gt_torch)
    exact = None
    if args.impl == "ours" and rank == 0:
        qbf = gen_set(nq, dim, base_seed + 3000, dev).cpu().numpy()
        ix.bruteforce(qbf, k)
        t0 = time.perf_counter()
        _, _, st = ix.bruteforce(qbf, k, stats=True)
        bf_s = time.perf_counter() - t0
        tf = 2.0 * nq * n * dim / (st["gemm_ms"] * 1e-3) / 1e12
        tr = measured_traffic("exact_scan", rows=n, dim=dim, queries=nq)
        exact = {"queries_per_s": round(nq / bf_s, 1), "gemm_ms": round(st["gemm_ms"], 3), "gemm_tflops": round(tf, 1),
                 # one GEMM launch timed alone: the burst figure of MEASURED_PEAKS.json is the denominator
                 "tensor_peak_tflops": bf16_peak, "peak_kind": peak_kind + " (bf16_tflops, burst: one kernel timed alone)",
                 "frac_of_tensor_peak": round(tf / bf16_peak, 4),
                 "certified_exact": st["certified"], "rescanned_fp32": st["rescanned"], "batch": nq,
                 "agreement_with_torch_fp32_top10": round(gt_agree, 5),
                 "ncu": tr}
    torch.cuda.empty_cache()
    stream = torch.cuda.current_stream().cuda_stream
    efs = [args.ef] if args.ef > 0 else [40, 50, 60, 70, 80, 90, 100, 120, 150, 200, 300, 400]
    ef, rec, sweep = pick_ef(ix, q_eval, gt, nq_eval, efs, stream, torch)
    log("[rank %d] ef_search=%d recall@10=%.4f sweep=%s" % (rank, ef, rec, sweep))

    if args.impl == "reference":
        return run_reference(args, ix, q_eval, ef, rec, n, dim, nq)

    q_all = gen_set(nq * total_steps, dim, base_seed + 2000 + rank, dev).view(total_steps, nq, dim)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident steps
    # Steps rotate over three CUDA streams (each with its own output buffers), the way a server keeps
    # batches in flight: the drain of one batch overlaps the ramp of the next.
    streams = [torch.cuda.Stream(device=dev) for _ in range(NSLOT)]
    outs = [(torch.empty((nq, ef), dtype=torch.int32, device=dev), torch.empty((nq, ef), dtype=torch.float32, device=dev),
             torch.empty((nq,), dtype=torch.int32, device=dev)) for _ in range(NSLOT)]
    main = torch.cuda.current_stream(dev)

    def run_steps(first, count):
        for st in streams:
            st.wait_stream(main)
        for s in range(count):
            st, (e_, d_, c_) = streams[s % NSLOT], outs[s % NSLOT]
            ix.search_dev(q_all[first + s].data_ptr(), nq, ef, e_.data_ptr(), d_.data_ptr(), c_.data_ptr(), st.cuda_stream)
        for st in streams:
            main.wait_stream(st)

    run_steps(0, args.warmup)
    torch.cuda.synchronize()
    ix.counters(reset=True)
    clocks = ClockSampler(local_rank)
    time.sleep(0.3)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(main)
    run_steps(args.warmup, args.steps)
    ev1.record(main)
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    ctr = ix.counters(reset=True)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        # before the single launch below, which writes slot 0 again
        dump_outputs(args.dump_outputs, dict(zip(("elements", "distances", "counts"),
                                                 (t.cpu().numpy() for t in outs[(args.steps - 1) % NSLOT]))))
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        total_ms = float(t.item())
    qps = world * nq * args.steps / (total_ms / 1e3)

    # one launch on its own (library events around the scan kernels on their stream): the un-pipelined figure
    ix.search_dev(q_all[0].data_ptr(), nq, ef, outs[0][0].data_ptr(), outs[0][1].data_ptr(), outs[0][2].data_ptr(), streams[0].cuda_stream)
    torch.cuda.synchronize()
    single_launch_ms = ix.last_search_ms()
    ix.counters(reset=True)

    # algorithmic bytes (SURVEY.md 8d): distance evaluations x row + neighbour lists + the query
    alg_bytes = (ctr["n_dist"] * row_bytes + ctr["n_hop0"] * (2 * 16 * 4) + ctr["n_hopu"] * (16 * 4) + nq * args.steps * row_bytes)
    alg_per_launch = alg_bytes / args.steps
    ms_per_step = total_ms / args.steps
    achieved = alg_per_launch / (ms_per_step / 1e3) / 1e9

    # ---------------------------------------------------------------- end to end through the C ABI
    # host (pinned) buffers in and out; three batches in flight (hb_search_batch_async slots), so every
    # step's H2D copy, scan and D2H read are inside the timed region and overlap one another.
    qh = torch.empty((total_steps, nq, dim), dtype=torch.float32).pin_memory()
    qh.copy_(q_all.cpu())
    houts = [(torch.empty((nq, k), dtype=torch.int64).pin_memory(), torch.empty((nq, k), dtype=torch.float32).pin_memory(),
              torch.empty((nq,), dtype=torch.int32).pin_memory()) for _ in range(NSLOT)]

    def run_e2e(first, count):
        for s in range(count):
            slot = s % NSLOT
            ix.search_wait(slot)
            t_, d_, c_ = houts[slot]
            ix.search_async(slot, qh[first + s].data_ptr(), nq, k, ef, t_.data_ptr(), d_.data_ptr(), c_.data_ptr())
        for slot in range(NSLOT):
            ix.search_wait(slot)

    run_e2e(0, args.warmup)
    barrier()
    t0 = time.perf_counter()
    run_e2e(args.warmup, args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_qps = world * nq * args.steps / e2e_s
    e2e_recall = None
    if rank == 0:
        out_t, out_d, out_c = houts[0]
        ix.search_into(q_eval.cpu().pin_memory().data_ptr(), nq_eval, k, ef, out_t.data_ptr(), out_d.data_ptr(), out_c.data_ptr())
        e2e_recall = recall_at(out_t[:nq_eval].numpy(), gt)
    del qh, q_all

    # ---------------------------------------------------------------- CPU baseline + full-size parity (rank 0, N = 1)
    cpu, parity, build_cpu = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            q_eval_host = q_eval.cpu().numpy()
            res, par = cpu_search_arm(ix, q_eval_host, ef, args.steps, args.warmup, args.cpu_budget, parity=nq_eval,
                                      build_rows=x_host[:min(n, 100000)],
                                      build_meta={"metric": 2, "dtype": 0, "m": 16, "efc": 64, "n1": 20000, "parts": 0, "n_part": 10000})
            cpu = cpu_baseline_record(res, nq, ef)
            build_cpu = res.get("build")
            e_ = torch.empty((nq_eval, ef), dtype=torch.int32, device=dev)
            d_ = torch.empty((nq_eval, ef), dtype=torch.float32, device=dev)
            c_ = torch.empty((nq_eval,), dtype=torch.int32, device=dev)
            ix.counters(reset=True)
            ix.search_dev(q_eval.data_ptr(), nq_eval, ef, e_.data_ptr(), d_.data_ptr(), c_.data_ptr(), stream)
            torch.cuda.synchronize()
            parity = parity_record(par, e_.cpu().numpy(), d_.cpu().numpy())
            c1 = ix.counters(reset=True)
            parity["counters_identical"] = all(int(c1[kk]) == int(res["canon_counters"][kk]) for kk in ("n_dist", "n_hop0", "n_hopu"))
        except Exception as e:   # the baseline is reported, never required
            cpu = {"error": str(e)[:300]}
    del x_host

    line = None
    if rank == 0:
        tr = measured_traffic("scan", rows=n, dim=dim, queries=nq, ef_search=ef)
        build_tr = measured_traffic("build", rows=n, dim=dim)
        line = {
            "metric": "QPS @ recall@10>=0.95 (1M x 768 cosine)", "value": round(qps, 1), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_C2 % (n, dim, ef, nq),
                       "batching": "batches resident in HBM, steps rotate over %d streams%s" % (NSLOT, "" if world == 1 else ", one replica per GPU (replicas only)"),
                       "ef_search": ef, "recall@10": round(rec, 4), "recall_sweep": sweep, "parallelism": "replicas x%d" % world,
                       "l2_policy": "inputs larger than L2: graph+vectors %.2f GB, a distinct query batch every step" % ((n * row_bytes + n * 128) / 1e9),
                       "parity": "unpinned (reference mount has no source); see the parity key for GPU vs oracle on this graph"},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                         "frac": round(achieved / hbm_peak, 4),
                         # dram__bytes_read.sum + dram__bytes_write.sum of one scan_kernel launch of this exact workload,
                         # from the round's ncu --set full capture (profiles/traffic.json names the report and commit)
                         "traffic": tr["dram_bytes"] if tr else None, "traffic_source": tr.get("source") if tr else None,
                         # the same launch's measured DRAM bytes over this run's step time: what HBM actually moved
                         "dram_gbs": round(tr["dram_bytes"] / (ms_per_step / 1e3) / 1e9, 1) if tr else None,
                         "dram_frac": round(tr["dram_bytes"] / (ms_per_step / 1e3) / 1e9 / hbm_peak, 4) if tr else None,
                         "peak_kind": peak_kind,
                         "frac_of_nominal_8000": round(achieved / 8000.0, 4),
                         "algorithmic_bytes_per_launch": int(alg_per_launch), "kernel": "scan_kernel (batched HnswSearchLayer)",
                         "timing": "CUDA events around the %d pipelined steps; single_launch_ms = one launch alone on its stream" % args.steps,
                         "single_launch_ms": round(single_launch_ms, 4),
                         "single_launch_frac": round(alg_per_launch / (single_launch_ms / 1e3) / 1e9 / hbm_peak, 4),
                         "n_dist_per_query": round(ctr["n_dist"] / (nq * args.steps), 1),
                         "n_hop_per_query": round((ctr["n_hop0"] + ctr["n_hopu"]) / (nq * args.steps), 1),
                         "slow_path_queries": ctr["n_slow"]},
            "cpu_baseline": cpu,
            "parity": parity,
            "e2e": {"value": round(e2e_qps, 1), "unit": "queries/s", "h2d_bytes_per_step": nq * row_bytes,
                    "d2h_bytes_per_step": nq * (k * 12 + 4), "recall@10": e2e_recall},
            "exact_scan": exact,
            "gpu_launches": 3 * args.steps,
            "clocks": clk,
            "build": {"vectors_per_s": round(n_indexed / build_s, 1), "seconds": round(build_s, 2), "n": n_indexed,
                      "n_dist_per_insert": round(bc["n_dist"] / max(n_indexed, 1), 1), "n_pair_per_insert": round(bc["n_pair"] / max(n_indexed, 1), 1),
                      # measured DRAM bytes of all build kernels of one build (ncu), not the sequential algorithm's count:
                      # the link phase memoises pair distances, so algorithmic bytes would exceed what is fetched
                      "traffic": build_tr["dram_bytes"] if build_tr else None,
                      "achieved_gbs": round(build_tr["dram_bytes"] / build_s / 1e9, 1) if build_tr else None,
                      "frac_of_hbm_peak": round(build_tr["dram_bytes"] / build_s / 1e9 / hbm_peak, 4) if build_tr else None,
                      "traffic_source": build_tr.get("source") if build_tr else None,
                      "cpu_baseline": build_cpu},
        }
    ix.close()
    del ix
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- configs[2] and configs[3] at this N
    if not args.no_sub:
        part = run_partitioned(args, ctx, args.part_rows, 128)
        bpart = run_build_partitioned(args, ctx, args.build_rows, 1536)
        if rank == 0:
            line["partitioned"] = part
            line["build_partitioned"] = bpart
    if rank == 0:
        emit(line)
    return finish(torch, world)


def finish(torch, world):
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


def standalone_line(rec, world, args):
    line = {"metric": rec["metric"], "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": rec.get("steps", 1),
            "warmup": rec.get("warmup", 0), "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": rec["dtype"], "data": "synthetic", "config": {"workload": rec["workload"], "parallelism": rec["parallelism"]},
            "roofline": rec.get("roofline"), "e2e": rec.get("e2e"), "gpu_launches": rec.get("gpu_launches")}
    line.update({k: v for k, v in rec.items() if k not in line and k not in ("workload", "parallelism")})
    return line


def run_reference(args, ix, q_eval, ef, rec, n, dim, nq):
    """--impl reference: the CPU oracle in the child process, timed over bounded samples, all host threads."""
    import torch
    q_host = q_eval.cpu().numpy()
    d = shm_dir()
    try:
        write_graph_image(ix, d)
        ix.close()
        torch.cuda.empty_cache()
        np.save(os.path.join(d, "queries.npy"), q_host)
        res = run_cpu_child({"graph_dir": d, "queries": os.path.join(d, "queries.npy"), "ef": ef, "steps": args.steps,
                             "warmup": args.warmup, "budget_s": max(args.cpu_budget, 30.0), "threads": 0, "parity": 0}, d)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    qps = res["queries_per_s"]
    cb = cpu_baseline_record(res, nq, ef)
    line = {"impl": "reference", "metric": "QPS @ recall@10>=0.95 (1M x 768 cosine)", "value": round(qps, 1), "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(res["ms_per_step"], 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_C2 % (n, dim, ef, nq),
                       "batching": "each step a bounded sample of the batch: %d queries on %d host threads" % (res["per_step"], res["threads"]),
                       "ef_search": ef, "recall@10": round(rec, 4),
                       "graph_built_by": "hb_build on the GPU in the parent's untimed set-up; flat image handed to the child through /dev/shm",
                       "timed_process": "child (oracle/cpu_arm.py): numpy + oracle/libhnsw_oracle.so only, CUDA_VISIBLE_DEVICES empty",
                       "note": "CPU restatement of pgvector HNSW semantics (oracle/), not pgvector: the reference mount has no "
                               "source and the image has no PostgreSQL."},
            "cpu_baseline": cb,
            "e2e": {"value": round(qps, 1), "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------------
def owned_rows(pkg, torch, x_dev, P, rank, world):
    """rows (and heap TIDs = row numbers) of the partitions this rank owns, as host arrays"""
    n = x_dev.shape[0]
    tids = np.arange(n, dtype=np.int64)
    part = pkg.partition_route(tids, P)
    mine = np.nonzero(part % world == rank)[0]
    idx = torch.from_numpy(mine).to(x_dev.device)
    return x_dev[idx].cpu().numpy(), mine.astype(np.int64)


def run_partitioned(args, ctx, n, dim):
    """configs[2]: P hash partitions over the ranks (hb_part_*), queries resident on every rank (value) or
    broadcast from rank 0's host memory (e2e), one ncclAllGather of the per-rank top-k, merge.  Three batches
    in flight.  Strong scaling: the same 10 000-query batches at every N."""
    pkg, torch, dev, rank, local_rank, world = ctx["pkg"], ctx["torch"], ctx["dev"], ctx["rank"], ctx["local_rank"], ctx["world"]
    hbm_peak = ctx["hbm_peak"]
    nq, k, P = args.nq, 10, args.partitions
    ef = 40
    steps, warmup = args.steps, args.warmup
    opclass = "vector_l2_ops" if dim == 128 else "vector_cosine_ops"
    pix = pkg.PartitionedIndex(dim, opclass, P, 16, 64, capacity_per_partition=int(n / P * 1.1) + 1024, rank=rank, world=world,
                               device=local_rank, seed=3)
    x_dev = gen_set(n, dim, 20260103, dev)
    q_eval = gen_set(1000, dim, 20260103 + 500, dev)
    gt = exact_topk_metric(x_dev, q_eval, k, "l2" if dim == 128 else "cosine")
    x, tids = owned_rows(pkg, torch, x_dev, P, rank, world)
    del x_dev
    torch.cuda.empty_cache()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pix.build(x, tids)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    del x
    for ix in pix.parts.values():
        ix.trim()
    te, _ = pix.search_dev(q_eval, k, ef)
    rec = recall_at(te.cpu().numpy(), gt)
    pix.counters(reset=True)
    total_steps = warmup + steps
    q_all = gen_set(nq * total_steps, dim, 20260103 + 1000, dev).view(total_steps, nq, dim)   # same on every rank = already broadcast
    NSLOT = int(os.environ.get("HB_BENCH_PART_SLOTS", "4"))       # batches in flight (at most HB_PART_SLOTS = 4)
    outs = [(torch.empty((nq, k), dtype=torch.int64, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev)) for _ in range(NSLOT)]
    torch.cuda.synchronize()

    def run(first, count):
        for s in range(count):
            slot = s % NSLOT
            pix.search_wait(slot)
            pix.search_async(slot, q_all[first + s].data_ptr(), nq, k, ef, outs[slot][0].data_ptr(), outs[slot][1].data_ptr(),
                             root=-1, q_on_device=True, out_on_device=True)
        for slot in range(NSLOT):
            pix.search_wait(slot)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # every slot in flight is warmed (its buffers are sized on first use): with fewer warm-up steps than slots a
    # cudaMalloc would land inside the timed region
    run(0, max(warmup, min(NSLOT, total_steps)))
    pix.counters(reset=True)
    barrier()
    # the library runs on its own streams; the device is idle at both records, so the events bracket the steps
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    run(warmup, steps)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    c = pix.counters(reset=True)
    row_bytes = dim * 4
    alg = c["n_dist"] * row_bytes + c["n_hop0"] * 128 + c["n_hopu"] * 64 + len(pix.owned) * nq * steps * row_bytes
    tt = torch.tensor([ms, 0.0, float(alg), build_s], device=dev, dtype=torch.float64)
    # ---- end to end: host queries on rank 0 only, ncclBroadcast, results to every rank's host memory
    qh = q_all.cpu().pin_memory() if rank == 0 else None
    houts = [(torch.empty((nq, k), dtype=torch.int64).pin_memory(), torch.empty((nq, k), dtype=torch.float32).pin_memory()) for _ in range(NSLOT)]

    def run_e2e(first, count):
        for s in range(count):
            slot = s % NSLOT
            pix.search_wait(slot)
            pix.search_async(slot, qh[first + s].data_ptr() if rank == 0 else 0, nq, k, ef, houts[slot][0].data_ptr(),
                             houts[slot][1].data_ptr(), root=0 if world > 1 else -1)
        for slot in range(NSLOT):
            pix.search_wait(slot)

    run_e2e(0, max(warmup, min(NSLOT, total_steps)))
    barrier()
    t0 = time.perf_counter()
    run_e2e(warmup, steps)
    torch.cuda.synchronize()
    tt[1] = time.perf_counter() - t0
    last_t = houts[(steps - 1) % NSLOT][0].numpy().copy()
    same = bool((last_t == outs[(steps - 1) % NSLOT][0].cpu().numpy()).all())
    if world > 1:
        tmax = tt.clone()
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.SUM)
        ms, e2e_s, build_s = float(tmax[0]), float(tmax[1]), float(tmax[3])
    else:
        e2e_s = float(tt[1])
    alg_total = float(tt[2])
    gbs_per_gpu = alg_total / (ms / 1e3) / 1e9 / world
    pix.close()
    del q_all
    torch.cuda.empty_cache()
    own = len([p for p in range(P) if p % world == rank])
    return {"metric": "QPS (hash-partitioned, %d partitions, merged top-%d)" % (P, k), "value": round(nq * steps / (ms / 1e3), 1), "unit": "queries/s",
            "steps": steps, "warmup": warmup, "ms_per_step": round(ms / steps, 4), "scaling": "strong", "dtype": "f32",
            "workload": "%s: %dx%d fp32 L2 in %d hash partitions, m=16, ef_construction=64, ef_search=%d, k=10, %d queries/step, "
                        "queries on every rank, one ncclAllGather of per-rank top-k + merge"
                        % ("configs[2]" if (n, dim, P) == (10000000, 128, 8) else "configs[2]-shaped, reduced", n, dim, P, ef, nq),
            "parallelism": "partitions/%d (hb_part_*, %d batches in flight)" % (world, NSLOT), "ef_search": ef, "recall@10": round(rec, 4),
            "roofline": {"bound": "hbm", "achieved": round(gbs_per_gpu, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(gbs_per_gpu / hbm_peak, 4),
                         "traffic": None, "note": "per GPU, algorithmic bytes from the in-kernel counters; every query visits every partition"},
            "e2e": {"value": round(nq * steps / e2e_s, 1), "unit": "queries/s", "h2d_bytes_per_step": nq * row_bytes,
                    "d2h_bytes_per_step": world * nq * k * 12, "note": "host queries on rank 0, ncclBroadcast, results copied to every rank's host memory",
                    "same_answer_as_resident_path": same},
            "build": {"seconds": round(build_s, 2), "vectors_per_s": round(n / build_s, 1)},
            "gpu_launches": steps * (own * 4 + 2)}


def run_build_partitioned(args, ctx, n, dim):
    """configs[3]: HNSW index build, 1M x 1536 halfvec inner product, hash-partitioned into P partitions that the
    ranks build independently (hb_part_build, no collective); then a merged search at ef_search=40 checks recall of
    what was built.  value = rows / max-over-ranks build time."""
    pkg, torch, dev, rank, local_rank, world = ctx["pkg"], ctx["torch"], ctx["dev"], ctx["rank"], ctx["local_rank"], ctx["world"]
    hbm_peak = ctx["hbm_peak"]
    k, P = 10, args.partitions
    opclass = os.environ.get("HB_BUILD_OPCLASS", "halfvec_ip_ops")
    half = opclass.startswith("halfvec")
    metric = "ip" if "_ip_" in opclass else ("l2" if "_l2_" in opclass else "cosine")
    x = gen_set(n, dim, 20260104, dev)
    if metric == "ip":     # not normalised: norms ~ lognormal(sigma = 0.1)
        x = x * torch.exp(0.1 * torch.randn((n, 1), device=dev, generator=torch.Generator(device=dev).manual_seed(5)))
    xs = x.half() if half else x
    del x
    q = gen_set(1000, dim, 20260104 + 1000, dev)
    qs = q.half() if half else q
    gt = exact_topk_metric(xs, qs, k, metric)
    x_host, tids = owned_rows(pkg, torch, xs, P, rank, world)
    del xs
    torch.cuda.empty_cache()
    pix = pkg.PartitionedIndex(dim, opclass, P, 16, 64, capacity_per_partition=int(n / P * 1.1) + 1024, rank=rank, world=world,
                               device=local_rank, seed=3)
    warm = pkg.HnswIndex(dim, opclass, 16, 64, capacity=4096, device=local_rank, seed=3)     # loads the kernels' modules
    warm.build(x_host[:4096])
    warm.close()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pix.build(x_host, tids)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    c = pix.counters(reset=True)
    tt = torch.tensor([build_s, float(c["n_dist"]), float(c["n_pair"])], device=dev, dtype=torch.float64)
    if world > 1:
        tmax = tt.clone()
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.SUM)
        build_s = float(tmax[0].item())
    n_dist, n_pair = float(tt[1].item()), float(tt[2].item())
    t, d = pix.search_dev(qs, k, 40)
    rec = recall_at(t.cpu().numpy(), gt)
    pix.close()
    del x_host
    torch.cuda.empty_cache()
    tr = measured_traffic("build_partitioned", rows=n, dim=dim, n_gpus=world)
    return {"metric": "HNSW build vectors/s", "value": round(n / build_s, 1), "unit": "vectors/s", "steps": 1, "warmup": 0,
            "ms_per_step": round(build_s * 1e3, 1), "scaling": "strong", "dtype": "f16" if half else "f32",
            "workload": "configs[3]: %dx%d %s index build, m=16, ef_construction=64, %d hash partitions built independently by "
                        "%d rank(s), host rows in, no collective" % (n, dim, opclass, P, world),
            "parallelism": "partitions/%d (hb_part_build)" % world, "recall@10_ef40_merged": round(rec, 4),
            "n_dist_per_insert": round(n_dist / n, 1), "n_pair_per_insert": round(n_pair / n, 1),
            "roofline": {"bound": "hbm", "traffic": tr["dram_bytes"] if tr else None,
                         "achieved": round(tr["dram_bytes"] / build_s / 1e9 / world, 1) if tr else None, "peak": hbm_peak, "unit": "GB/s",
                         "frac": round(tr["dram_bytes"] / build_s / 1e9 / world / hbm_peak, 4) if tr else None,
                         "note": "measured DRAM bytes of the build kernels (ncu) / build seconds, per GPU; null without a capture of this shape. "
                                 "The sequential algorithm's (n_dist + n_pair) x row is NOT used: the link phase memoises pair distances"},
            "gpu_launches": None}


if __name__ == "__main__":
    sys.exit(main())
