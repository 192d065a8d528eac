"""bench.py's contract where it can be checked without a GPU: the reference arm answers with one JSON line and
exit code 0, the product arm refuses to run (no CPU fallback), the helpers behave."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def has_cuda():
    import torch
    return torch.cuda.is_available()


def test_reference_arm_without_gpu_prints_one_json_line():
    if has_cuda():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and "unavailable" in d


def test_product_arm_without_gpu_fails_loudly():
    if has_cuda():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and out.stdout.strip() == ""
    assert "no CPU fallback" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, timeout=300, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_recall_helper():
    sys.path.insert(0, ROOT)
    import bench
    ids = np.array([[1, 2, 3, 4], [5, 6, 7, 8]])
    gt = np.array([[1, 2, 9, 10], [5, 6, 7, 8]])
    assert bench.recall_at(ids, gt) == 0.75


def test_cpu_arm_child_process(tmp_path):
    """oracle/cpu_arm.py (the process whose time bench.py reports as the CPU arm): loads a flat graph image,
    times bounded steps, returns the ids both summation orders give; it imports neither torch nor the product."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import oracle as O
    from conftest import clustered
    src = open(os.path.join(ROOT, "oracle", "cpu_arm.py")).read()
    assert "import torch" not in src and "pgvector_hnsw_partitioning_b200" not in src and "libhnsw_b200" not in src
    x = clustered(3000, 32, 16, seed=4)
    q = clustered(200, 32, 16, seed=5)
    orc = O.Index(32, 16, 64, O.COSINE, O.F32, O.CANON, seed=3)
    orc.build(x)
    g = orc.export()
    d = str(tmp_path)
    for k in ("vecs", "level", "nbr0", "uoff", "nbru", "ntids", "tids"):
        np.save(os.path.join(d, k + ".npy"), getattr(g, k))
    json.dump({"dim": g.dim, "m": g.m, "efc": g.efc, "metric": g.metric, "dtype": g.dtype, "n": g.n, "upper_rows": g.upper_rows,
               "entry": g.entry}, open(os.path.join(d, "meta.json"), "w"))
    np.save(os.path.join(d, "queries.npy"), q)
    np.save(os.path.join(d, "rows.npy"), x)
    job = {"graph_dir": d, "queries": os.path.join(d, "queries.npy"), "ef": 40, "steps": 3, "warmup": 1, "budget_s": 1.0, "threads": 2,
           "parity": 100, "parity_out": os.path.join(d, "parity.npz"),
           "build": {"rows": os.path.join(d, "rows.npy"), "metric": 2, "dtype": 0, "n1": 500, "parts": 2, "n_part": 300}}
    res = bench.run_cpu_child(job, d)
    assert res["kind"] == "port" and res["queries_per_s"] > 0 and res["threads"] == 2 and 64 <= res["per_step"] <= 200
    assert res["build"]["single_thread"]["vectors_per_s"] > 0 and res["build"]["concurrent"]["partitions"] == 2
    par = dict(np.load(os.path.join(d, "parity.npz")))
    oe, od, oc, octr = orc.search_batch(q[:100], 40, threads=2)
    assert (par["canon_ids"] == oe).all() and (par["canon_dist"].view(np.uint32) == od.view(np.uint32)).all()
    assert res["canon_counters"]["n_dist"] == octr["n_dist"]
    # the parity record: identical ids -> everything identical; a perturbed id that is not a tie -> unexplained
    rec = bench.parity_record(par, oe.copy(), od.copy())
    assert rec["canonical_order"]["ids_identical"] == 100 and rec["canonical_order"]["distances_bit_identical"] == 100
    nat = rec["natural_order_top10"]
    assert nat["ids_identical"] + nat["within_1e-5_ties"] == 100 and nat["unexplained"] == 0
    bad = oe.copy()
    bad[0, 0] = oe[0, 20]
    bd = od.copy()
    bd[0, 0] = od[0, 20]
    rec2 = bench.parity_record(par, bad, bd)
    assert rec2["canonical_order"]["ids_identical"] == 99 and rec2["natural_order_top10"]["unexplained"] == 1


def test_dump_outputs_writes_float_arrays_and_samples_above_the_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    elem = np.arange(60, dtype=np.int32).reshape(20, 3)
    elem[4, 2] = -1
    dist = (elem / 7).astype(np.float32)
    dist[4, 2] = np.inf
    arrays = {"elements": elem, "distances": dist, "counts": np.full(20, 3, np.int32)}
    d = str(tmp_path / "all")
    bench.dump_outputs(d, arrays)
    got = {k: np.load(os.path.join(d, k + ".npy")) for k in ("elements", "distances", "counts", "rows")}
    assert got["elements"].dtype == np.float64 and got["counts"].dtype == np.float64 and got["distances"].dtype == np.float32
    assert (got["rows"] == np.arange(20)).all() and (got["elements"] == elem).all() and (got["counts"] == 3).all()
    assert (got["distances"].view(np.uint32) == dist.view(np.uint32)).all()
    # 52 bytes a row (rows + 3 ids + 3 distances + count) and 1 kB per header: room for 10 of the 20 rows
    limit = 4 * 1024 + 52 * 10
    picks = []
    for tag in ("a", "b"):
        d = str(tmp_path / tag)
        bench.dump_outputs(d, arrays, limit=limit)
        rows = np.load(os.path.join(d, "rows.npy")).astype(np.int64)
        assert len(rows) == 10 and (np.diff(rows) > 0).all()
        assert (np.load(os.path.join(d, "elements.npy")) == elem[rows]).all()
        assert (np.load(os.path.join(d, "distances.npy")).view(np.uint32) == dist[rows].view(np.uint32)).all()
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= limit
        picks.append(rows)
    assert (picks[0] == picks[1]).all()


def test_dump_outputs_is_refused_outside_the_headline_scan(tmp_path):
    for extra in (["--impl", "reference"], ["--workload", "build"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path)] + extra,
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 2 and "--dump-outputs" in out.stderr and out.stdout == ""
