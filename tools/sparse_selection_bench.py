"""Cross-validation of sparse input on one B200, at the Netflix shape: where the time and the memory of a run go.

    python tools/sparse_selection_bench.py [--out profiles/r09_sparse_selection_bench.json] [--iterations 100] [--folds 5]

Data: 480 189 x 17 770 with 100 480 507 stored entries, at least 20 in every row and every column (the reference's fold
rule needs them: a row with n entries empties one of f training masks with probability about f^(1-n), so with a few
entries per row over 10^5 rows no split ever passes), then seeded power-law row and column lengths as in
tools/sparse_bench.py, values from a seeded rank-20 model plus noise, raised to at least 0.01.

Runs, one after the other, each from numpy / random seed 0:
  lscv : LineSearchCrossValidation(bnmf_vb_optimised, values_K=[10, 20], folds, iterations, restarts=1, 'AIC')
  mcv  : MatrixCrossValidation(NMF, folds, [{'K': 20}], iterations)
For each: the wall time of the whole run and of its parts -- the fold split (the python shuffle and the fold checks; the
shuffle alone and the host memory it adds), each fold's SparseDataset build, the fits (the rest), the test-fold
predictions -- the host peak RSS, the device memory high-water mark, and the fold-build share (fold split + dataset
builds over the whole run).  Every part ends in a device synchronise.  Prints one JSON line and writes it to --out.
"""
import argparse
import importlib.util
import json
import os
import resource
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _sparse_bench():
    spec = importlib.util.spec_from_file_location("sparse_bench", os.path.join(ROOT, "tools", "sparse_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def rss_bytes():
    with open("/proc/self/status") as fh:
        for line in fh:
            if line.startswith("VmRSS:"):
                return int(line.split()[1]) * 1024
    return 0


def netflix_floor(sb, floor=20, seed=0, K=20, device="cuda"):
    """tools/sparse_bench.py's Netflix-shaped matrix with `floor` entries guaranteed in every row and column: `floor`
    consecutive columns (from a seeded start) in every row and `floor` consecutive rows in every column, then power-law
    pairs up to nnz; extras are dropped from the power-law pairs only."""
    import scipy.sparse as sp
    import torch
    I, J, nnz = sb.NETFLIX
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    rnd = lambda n: torch.rand(n, generator=gen, device=device, dtype=torch.float64)
    k = torch.arange(floor, device=device)
    c0 = torch.randint(0, J, (I, 1), generator=gen, device=device)
    r0 = torch.randint(0, I, (J, 1), generator=gen, device=device)
    base = torch.unique(torch.cat([(torch.arange(I, device=device)[:, None] * J + (c0 + k) % J).ravel(),
                                   (((r0 + k) % I) * J + torch.arange(J, device=device)[:, None]).ravel()]))
    ca, cb = sb._cdf(I, 0.8, 120.0, gen, device), sb._cdf(J, 1.0, 30.0, gen, device)
    draw = lambda c, n, m: torch.searchsorted(c, rnd(m)).clamp_(max=n - 1)
    keys = base
    while keys.numel() < nnz:
        m = int((nnz - keys.numel()) * 1.1) + 1024
        keys = torch.unique(torch.cat([keys, draw(ca, I, m) * J + draw(cb, J, m)]))
    if keys.numel() > nnz:
        extra = keys[~torch.isin(keys, base)]
        keep = torch.randperm(extra.numel(), generator=gen, device=device)[:nnz - base.numel()]
        keys = torch.sort(torch.cat([base, extra[keep]])).values
    rows, cols = keys // J, keys % J
    assert int(torch.bincount(rows, minlength=I).min()) >= floor and int(torch.bincount(cols, minlength=J).min()) >= floor
    U = -torch.log(rnd(I * K)).view(I, K)
    V = -torch.log(rnd(J * K)).view(J, K)
    vals = torch.empty(nnz, dtype=torch.float64, device=device)
    for t0 in range(0, nnz, 1 << 24):
        t1 = min(nnz, t0 + (1 << 24))
        vals[t0:t1] = (U[rows[t0:t1]] * V[cols[t0:t1]]).sum(1) / K
    vals += 0.25 * torch.randn(nnz, generator=gen, device=device, dtype=torch.float64)
    vals.clamp_(min=0.01)
    indptr = torch.cat([torch.zeros(1, dtype=torch.int64, device=device), torch.cumsum(torch.bincount(rows, minlength=I), 0)])
    return sp.csr_matrix((vals.cpu().numpy(), cols.to(torch.int32).cpu().numpy(), indptr.cpu().numpy()), shape=(I, J))


class Timer:
    """Wraps functions so that each call is timed, up to a device synchronise, under a name."""

    def __init__(self):
        import torch
        self.torch, self.t, self.patched = torch, {}, []

    def wrap(self, owner, attr, name):
        real = getattr(owner, attr)
        torch, t = self.torch, self.t

        def timed(*a, **k):
            t0 = time.perf_counter()
            out = real(*a, **k)
            torch.cuda.synchronize()
            t.setdefault(name, []).append(time.perf_counter() - t0)
            return out
        setattr(owner, attr, timed)
        self.patched.append((owner, attr, real))

    def restore(self):
        for owner, attr, real in reversed(self.patched):
            setattr(owner, attr, real)
        self.patched = []


def run_one(name, build, dev):
    import random
    import torch
    from bnmtf_b200 import engine, mask, model_selection
    from bnmtf_b200.bnmf import bnmf_vb_optimised
    from bnmtf_b200.np_models import NMF
    tm = Timer()
    shuffle_rss = []
    real_shuffled = mask._shuffled

    def shuffled(n):
        r0 = rss_bytes()
        t0 = time.perf_counter()
        out = real_shuffled(n)
        tm.t.setdefault("shuffle_s", []).append(time.perf_counter() - t0)
        shuffle_rss.append(rss_bytes() - r0)
        return out
    mask._shuffled = shuffled
    tm.wrap(mask, "_fold_selections_attempts", "fold_split_s")
    tm.wrap(model_selection, "_cv_folds", "folds_with_test_masks_s")
    tm.wrap(engine.SparseDataset, "__init__", "dataset_build_s")
    for cls in (bnmf_vb_optimised, NMF):
        tm.wrap(cls, "predict", "predict_s")
    np.random.seed(0)
    random.seed(0)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.perf_counter()
    try:
        cv = build()
        cv.run()
        torch.cuda.synchronize()
    finally:
        tm.restore()
        mask._shuffled = real_shuffled
    total = time.perf_counter() - t0
    s = {k: float(np.sum(v)) for k, v in tm.t.items()}
    ds = tm.t.get("dataset_build_s", [])
    out = {"wall_s": total, "fold_split_s": s.get("fold_split_s", 0.0), "shuffle_s": tm.t.get("shuffle_s", []),
           "shuffle_rss_added_bytes": shuffle_rss, "test_masks_s": s.get("folds_with_test_masks_s", 0.0) - s.get("fold_split_s", 0.0),
           "dataset_builds": len(ds), "dataset_build_s": ds, "predict_s": tm.t.get("predict_s", []),
           "host_peak_rss_GB": resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024 / 1e9,
           "device_peak_GB": torch.cuda.max_memory_allocated(dev) / 1e9}
    build_s = out["fold_split_s"] + out["test_masks_s"] + sum(ds)
    out["fits_s"] = total - build_s - sum(out["predict_s"])
    out["fold_build_share"] = build_s / total
    cv.fout.close()
    print(json.dumps({name: out}), file=sys.stderr, flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iterations", type=int, default=100)
    ap.add_argument("--folds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    import torch
    from bnmtf_b200 import NMF, bnmf_vb_optimised, model_selection as ms
    sb = _sparse_bench()
    dev = torch.device("cuda", 0)
    res = {"gpu": sb.gpu_info(), "iterations": args.iterations, "folds": args.folds}
    t0 = time.perf_counter()
    R = netflix_floor(sb, seed=args.seed, device=dev)
    torch.cuda.empty_cache()
    res.update({"shape": list(R.shape), "nnz": int(R.nnz), "data_s": time.perf_counter() - t0,
                "min_per_row": int(np.diff(R.indptr).min()), "min_per_column": int(np.bincount(R.indices, minlength=R.shape[1]).min())})
    tmp = tempfile.mkdtemp()
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
    res["lscv_vb"] = run_one("lscv_vb", lambda: ms.LineSearchCrossValidation(
        bnmf_vb_optimised, R, None, [10, 20], args.folds, pri, 'random', args.iterations, 1, 'AIC',
        os.path.join(tmp, "lscv.txt"), devices=1), dev)
    res["mcv_nmf"] = run_one("mcv_nmf", lambda: ms.MatrixCrossValidation(
        NMF, R, None, args.folds, [{"K": 20}], {"iterations": args.iterations, "init_UV": "random"},
        os.path.join(tmp, "mcv.txt"), devices=1), dev)
    log = open(os.path.join(tmp, "mcv.txt")).read()
    assert "Average performances" in log and "exception" not in log, log
    res["mcv_nmf"]["log_tail"] = log[-300:]
    res["power_state_after"] = sb.gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
