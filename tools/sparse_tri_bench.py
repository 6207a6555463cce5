"""Sparse input of the tri-factor models at the Netflix shape (one B200): sweeps/s of VB, Gibbs and ICM, the CUDA-event
time of every call of a sweep, the K-means initialisation of F and G, and the device memory high-water mark.

    python tools/sparse_tri_bench.py [--out profiles/r07_sparse_tri_bench.json] [--KL 10 20] [--min-seconds 2.5]

The matrix is tools/sparse_bench.py's netflix_like(): 480 189 x 17 770 with 100 480 507 observed entries.  Per-call times
come from eager sweeps (no CUDA graph) with a pair of CUDA events around every library call, so they add up to a little
more than a replayed sweep; `S_phase_share` is the S-phase reduction (bnmtf_nmtf_sq_f64) over the whole sweep's calls.
Prints one JSON line, and writes it to --out.
"""
import argparse
import importlib.util
import json
import os
import random
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# library call -> the step of the sweep it is
STEP = {"bnmtf_csr_stats_f64": "stats", "bnmtf_nmtf_transform_f64": "transform", "bnmtf_nmtf_sq_f64": "S_reduction",
        "bnmtf_coord_solve_f64": "coord_solve", "bnmf_row_solve_f64": "row_solve", "bnmtf_nmtf_mstat_f64": "metrics",
        "bnmtf_mstat_reduce_f64": "metrics", "bnmtf_metrics_from_sums_f64": "metrics", "bnmtf_csr_metrics_f64": "metrics",
        "bnmtf_select_metrics_f64": "metrics", "bnmtf_small_matmul_f64": "metrics", "bnmtf_pad_factor_f64": "pad",
        "bnmtf_nmtf_extra_f64": "vb_terms", "bnmtf_reduce1_f64": "vb_terms", "bnmtf_vb_factor_terms_f64": "vb_terms",
        "bnmtf_reduce8_f64": "vb_terms", "bnmf_finish_sweep_f64": "finish"}


def _sparse_bench():
    spec = importlib.util.spec_from_file_location("sparse_bench", os.path.join(ROOT, "tools", "sparse_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def sweeps_per_s(model, min_seconds):
    """Sweeps per second of replayed sweeps (after a two-sweep warm-up run)."""
    import torch
    eng = model._engine()
    vb = eng.vb
    order = lambda: {"S": random.sample(range(eng.K * eng.L), eng.K * eng.L), "F": random.sample(range(eng.K), eng.K),
                     "G": random.sample(range(eng.L), eng.L)} if vb else None
    eng.alloc_trace(4096)                   # one trace window: the sweep graph is captured once and replayed
    for _ in range(3):
        eng.sweep(order=order())
    torch.cuda.synchronize()
    n, t0 = 0, time.perf_counter()
    while n + 10 <= 4093:
        for _ in range(10):
            eng.sweep(order=order())
        torch.cuda.synchronize()
        n += 10
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    return n / dt, n, dt, eng._graph is not None


def call_times(model, reps=3):
    """ms per sweep of every step (sum over its calls), and per call, from eager sweeps with events around each call."""
    import torch
    from bnmtf_b200 import _lib
    eng = model._engine()
    real = _lib.call
    rec = []

    def timed(name, *args):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = real(name, *args)
        e1.record()
        rec.append((name, e0, e1))
        return r
    K, L = eng.K, eng.L
    order = {"S": list(range(K * L)), "F": list(range(K)), "G": list(range(L))} if eng.vb else None
    _lib.call = timed
    try:
        eng.alloc_trace(reps)
        for _ in range(reps):
            eng._sweep_eager(0.0, order)
        torch.cuda.synchronize()
    finally:
        _lib.call = real
    steps, calls = {}, {}
    for name, a, b in rec:
        ms = a.elapsed_time(b) / reps
        steps[STEP.get(name, name)] = steps.get(STEP.get(name, name), 0.0) + ms
        calls.setdefault(name, []).append(ms)
    # the two statistics calls: row phase (rows of R against G), column phase (rows of R^T against F)
    st = [a.elapsed_time(b) for name, a, b in rec if name == "bnmtf_csr_stats_f64"]
    per = len(st) // reps
    out = {"steps_ms": steps, "total_ms": sum(steps.values()),
           "calls_ms": {k: [round(x, 4) for x in v[:len(v) // reps]] for k, v in calls.items()}}
    if per >= 2:
        out["stats_row_ms"] = float(np.mean(st[0::per]))
        out["stats_col_ms"] = float(np.mean(st[per - 1::per]))
    out["S_phase_share"] = steps.get("S_reduction", 0.0) / out["total_ms"]
    return out


def kmeans_times(ds, K, L, device):
    from bnmtf_b200.kmeans import SparseKMeans
    out = {}
    for side, X, Xall, k in (("F", ds.host_train, ds.host_R, K), ("G", ds.host_train.T.tocsr(), ds.host_R.T.tocsr(), L)):
        import torch
        random.seed(0)
        t0 = time.perf_counter()
        km = SparseKMeans(X, k, X_all=Xall, device=device)
        t1 = time.perf_counter()
        km.initialise()
        t2 = time.perf_counter()
        it = [0]
        real = km.assignment

        def counted():
            it[0] += 1
            return real()
        km.assignment = counted
        km.cluster()
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        out[side] = {"seconds": t3 - t0, "setup_s": t1 - t0, "initialise_s": t2 - t1, "cluster_s": t3 - t2,
                     "iterations": it[0], "points": km.no_points, "coordinates": km.no_coordinates,
                     "cluster_sizes": np.bincount(km.cluster_assignments, minlength=k).tolist()}
        del km
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--KL", type=int, nargs="+", default=[10, 20])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--min-seconds", type=float, default=2.5)
    ap.add_argument("--skip-kmeans", action="store_true")
    args = ap.parse_args()
    import torch
    import bnmtf_b200
    from bnmtf_b200 import data
    sb = _sparse_bench()
    dev = torch.device("cuda", 0)
    res = {"gpu": sb.gpu_info(), "power_state": sb.gpu_info()}
    R = sb.netflix_like(seed=args.seed, device=dev)
    torch.cuda.reset_peak_memory_stats(dev)
    ds = data.upload_sparse(R, device=dev)
    res.update({"shape": list(R.shape), "nnz": int(R.nnz), "device_csr_GB": ds.nbytes() / 1e9})
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaF": 0.1, "lambdaS": 0.1, "lambdaG": 0.1}
    classes = (("vb", bnmtf_b200.bnmtf_vb_optimised), ("gibbs", bnmtf_b200.bnmtf_gibbs_optimised),
               ("icm", bnmtf_b200.nmtf_icm))
    for KL in args.KL:
        r = {}
        for mode, cls in classes:
            np.random.seed(1), random.seed(1)
            m = cls.from_dataset(ds, KL, KL, pri, seed=1)
            m.initialise("random", "random")
            rate, n, dt, graph = sweeps_per_s(m, args.min_seconds)
            r[mode] = {"sweeps_per_s": rate, "sweeps": n, "seconds": dt, "graph_replayed": graph,
                       "sweep_ms": 1e3 / rate, "calls": call_times(m)}
            print(json.dumps({"K=L": KL, mode: r[mode]}), file=sys.stderr, flush=True)
            del m
        if not args.skip_kmeans:
            r["kmeans"] = kmeans_times(ds, KL, KL, dev)
            print(json.dumps({"K=L": KL, "kmeans": r["kmeans"]}), file=sys.stderr, flush=True)
        res["K%d" % KL] = r
    res["peak_device_GB"] = torch.cuda.max_memory_allocated(dev) / 1e9
    res["power_state_after"] = sb.gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
