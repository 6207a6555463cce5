"""Sparse input for the two-factor models on one GPU: the CSR statistics path (csrc/sparse.cu) at the Netflix shape, the
achieved rate of its statistics kernel, and the density at which the dense path overtakes it.

    python tools/sparse_bench.py [--out profiles/r05_sparse_bench.json] [--min-seconds 2.5] [--skip-density]

Prints one JSON line and writes it to --out.

  netflix : I = 480 189, J = 17 770, 100 480 507 observed entries (1.2 %), seeded power-law row and column lengths,
            values from a seeded non-negative rank-20 model plus noise (make_sparse).  K = 20: Gibbs and VB sweeps/s
            (each over >= --min-seconds), CUDA-event time of each statistics call (row phase, column phase), device memory
            high-water mark.  The dense layout of this matrix would take about 239 GB.
  rate    : FMAs (8x8 Gram tiles over the padded width KP, plus the R.X and variance sums) and bytes (the CSR streams plus
            the KP-wide factor rows gathered per entry) of one statistics call, counted from shapes, over its time.
  density : 65536 x 32768, K = 20, VB, both paths on the same seeded data at 0.5 .. 20 % observed: sweeps/s of each.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NETFLIX = (480189, 17770, 100480507)
PRI = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}


def _cdf(n, alpha, offset, gen, device):
    import torch
    w = (torch.arange(n, dtype=torch.float64, device=device) + offset) ** -alpha
    w = w[torch.randperm(n, generator=gen, device=device)]        # heavy rows / columns spread over the index range
    c = torch.cumsum(w, 0)
    return c / c[-1]


def make_sparse(I, J, nnz, seed=0, K=20, device="cuda", row_law=(0.8, 120.0), col_law=(1.0, 30.0), uniform=False):
    """A seeded I x J scipy CSR matrix with exactly nnz stored entries and no empty row or column.  Pattern: one entry per
    row and per column, then (row, column) pairs drawn from independent power laws w_i ~ (i + offset)^-alpha (uniform:
    equal weights), duplicates dropped, drawn again until nnz distinct pairs.  Values: U V^T + N(0, 0.25^2) with
    U ~ Exp(1), V ~ Exp(1) of rank K, evaluated at the stored entries only.  Generated with torch on `device`."""
    import scipy.sparse as sp
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    rnd = lambda n: torch.rand(n, generator=gen, device=device, dtype=torch.float64)
    ca = None if uniform else _cdf(I, row_law[0], row_law[1], gen, device)
    cb = None if uniform else _cdf(J, col_law[0], col_law[1], gen, device)
    draw = lambda c, n, m: (torch.searchsorted(c, rnd(m)).clamp_(max=n - 1) if c is not None
                            else torch.randint(0, n, (m,), generator=gen, device=device))
    keys = torch.cat([torch.arange(I, device=device) * J + torch.randint(0, J, (I,), generator=gen, device=device),
                      torch.randint(0, I, (J,), generator=gen, device=device) * J + torch.arange(J, device=device)])
    keys = torch.unique(keys)
    while keys.numel() < nnz:
        m = int((nnz - keys.numel()) * 1.1) + 1024
        keys = torch.unique(torch.cat([keys, draw(ca, I, m) * J + draw(cb, J, m)]))
    if keys.numel() > nnz:
        # drop random extras (the check below guards against a row or column losing its last entry)
        keep = torch.randperm(keys.numel(), generator=gen, device=device)[:nnz]
        keys = torch.sort(keys[keep]).values
    rows, cols = keys // J, keys % J
    assert int(torch.bincount(rows, minlength=I).min()) > 0 and int(torch.bincount(cols, minlength=J).min()) > 0, \
        "empty row or column: draw with another seed"
    U = -torch.log(rnd(I * K)).view(I, K)
    V = -torch.log(rnd(J * K)).view(J, K)
    vals = torch.empty(nnz, dtype=torch.float64, device=device)
    for t0 in range(0, nnz, 1 << 24):
        t1 = min(nnz, t0 + (1 << 24))
        vals[t0:t1] = (U[rows[t0:t1]] * V[cols[t0:t1]]).sum(1) / K
    vals += 0.25 * torch.randn(nnz, generator=gen, device=device, dtype=torch.float64)
    vals.clamp_(min=0.0)
    indptr = torch.cat([torch.zeros(1, dtype=torch.int64, device=device), torch.cumsum(torch.bincount(rows, minlength=I), 0)])
    return sp.csr_matrix((vals.cpu().numpy(), cols.to(torch.int32).cpu().numpy(), indptr.cpu().numpy()), shape=(I, J))


def netflix_like(seed=0, device="cuda"):
    return make_sparse(*NETFLIX, seed=seed, device=device)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def sweeps_per_s(model, min_seconds):
    """Sweeps per second of the device loop run() drives (the state stays on the device: no host transfers timed), from
    the third sweep on, i.e. replays of the captured sweep graph."""
    import torch
    model.run(2)
    eng = model._engine()
    torch.cuda.synchronize()
    n, t0 = 0, time.perf_counter()
    while True:
        eng.alloc_trace(10)
        for _ in range(10):
            eng.sweep()
        torch.cuda.synchronize()
        n += 10
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            return n / dt, n, dt


def stats_counts(ds, K, vb):
    """(FMAs, bytes) of one statistics call per phase, from shapes."""
    KP = 8 * ((K + 1 + 7) // 8)
    NT = KP // 8
    ntp = NT * (NT + 1) // 2
    out = {}
    for side, name, rows in ((0, "row", ds.I), (1, "col", ds.J)):
        n = ds.csr[side].nnz
        fma = n * (ntp * 64 + KP + (KP if vb else 0))                       # Gram tiles + r X + variance sums
        byts = n * (4 + 8) + 8 * (rows + 1) + n * KP * 8 * (2 if vb else 1) + rows * 8 * (ntp * 64 + KP * (2 if vb else 1))
        out[name] = (fma, byts)
    return out


def run_netflix(args, dev):
    import torch
    from bnmtf_b200 import bnmf, data
    t0 = time.perf_counter()
    R = netflix_like(seed=args.seed, device=dev)
    t_gen = time.perf_counter() - t0
    lens_r, lens_c = np.diff(R.indptr), np.bincount(R.indices, minlength=R.shape[1])
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.perf_counter()
    ds = data.upload_sparse(R, device=dev)
    torch.cuda.synchronize()
    t_up = time.perf_counter() - t0
    res = {"shape": list(R.shape), "nnz": int(R.nnz), "density": R.nnz / (R.shape[0] * R.shape[1]),
           "max_row_len": int(lens_r.max()), "max_col_len": int(lens_c.max()), "dense_layout_GB": R.shape[0] * R.shape[1] * 28 / 1e9,
           "device_csr_GB": ds.nbytes() / 1e9, "generate_s": t_gen, "upload_s": t_up, "K": args.K,
           "heavy_rows": {"row": ds.csr[0].n_heavy, "col": ds.csr[1].n_heavy}, "chunk": ds.csr[0].chunk}
    counts = stats_counts(ds, args.K, True)
    for mode, cls in (("vb", bnmf.bnmf_vb_optimised), ("gibbs", bnmf.bnmf_gibbs_optimised)):
        np.random.seed(1)
        m = cls.from_dataset(ds, args.K, PRI, seed=1)
        m.initialise("exp")
        rate, n, dt = sweeps_per_s(m, args.min_seconds)
        prof = m._engine().profile_sweep(reps=5)
        r = {"sweeps_per_s": rate, "sweeps": n, "seconds": dt, "stats_row_ms": prof["stats_csr_row"],
             "stats_col_ms": prof["stats_csr_col"], "row_solve_ms": prof["row_solve"],
             "graph_replayed": m._engine()._graph is not None, "MSE_after_2": m.all_performances["MSE"][-1]}
        vb = mode == "vb"
        c = stats_counts(ds, args.K, vb)
        for ph in ("row", "col"):
            fma, byts = c[ph]
            ms = r["stats_%s_ms" % ph]
            r["stats_%s_TFLOPs" % ph] = 2 * fma / (ms * 1e-3) / 1e12
            r["stats_%s_GBs" % ph] = byts / (ms * 1e-3) / 1e9
        res[mode] = r
        del m
    res["peak_device_GB"] = torch.cuda.max_memory_allocated(dev) / 1e9
    res["counts"] = {k: {"fma": v[0], "bytes": v[1]} for k, v in counts.items()}
    return res


def run_density(args, dev):
    """VB sweeps/s of the sparse and the dense path on the same seeded matrix at each density."""
    import scipy.sparse as sp
    import torch
    from bnmtf_b200 import bnmf, data, engine
    I, J = 65536, 32768
    out = []
    for pct in args.densities:
        nnz = int(round(pct / 100.0 * I * J))
        R = make_sparse(I, J, nnz, seed=args.seed + 7, device=dev, uniform=True)
        row = {"percent": pct, "nnz": nnz}
        ds = data.upload_sparse(R, device=dev)
        np.random.seed(1)
        m = bnmf.bnmf_vb_optimised.from_dataset(ds, args.K, PRI, seed=1)
        m.initialise("exp")
        row["sparse_sweeps_per_s"] = sweeps_per_s(m, args.min_seconds)[0]
        sp_mse = m.all_performances["MSE"][-1]
        del m, ds
        torch.cuda.empty_cache()
        # the same entries in the dense layout, built on the device (no host I x J array)
        ldJ = engine.ld_for(J)
        Rd = torch.zeros((I, ldJ), dtype=torch.float64, device=dev)
        rows = torch.repeat_interleave(torch.arange(I, device=dev), torch.from_numpy(np.diff(R.indptr)).to(dev))
        cols = torch.from_numpy(R.indices.astype(np.int64)).to(dev)
        Rd[rows, cols] = torch.from_numpy(R.data).to(dev)
        bitsw = torch.zeros((I, ldJ // 32), dtype=torch.int64, device=dev)
        bitsw.view(-1).index_add_(0, rows * (ldJ // 32) + cols // 32, (1 << (cols % 32)).to(torch.int64))
        bits = torch.where(bitsw >= 2 ** 31, bitsw - 2 ** 32, bitsw).to(torch.int32)
        del bitsw, rows, cols
        dd = engine.Dataset.from_device(Rd, bits, I, J, n_obs=nnz)
        np.random.seed(1)
        m = bnmf.bnmf_vb_optimised.from_dataset(dd, args.K, PRI, seed=1)
        m.initialise("exp")
        row["dense_sweeps_per_s"] = sweeps_per_s(m, args.min_seconds)[0]
        row["MSE_rel_diff"] = abs(m.all_performances["MSE"][-1] / sp_mse - 1)
        del m, dd, Rd, bits
        torch.cuda.empty_cache()
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    faster = [r["percent"] for r in out if r["dense_sweeps_per_s"] > r["sparse_sweeps_per_s"]]
    return {"shape": [I, J], "K": args.K, "rows": out, "dense_faster_from_percent": min(faster) if faster else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--K", type=int, default=20)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--min-seconds", type=float, default=2.5)
    ap.add_argument("--densities", type=float, nargs="+", default=[0.5, 1, 2, 5, 10, 20])
    ap.add_argument("--skip-density", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tools/sparse_bench.py measures on a GPU; none is visible")
    import __graft_entry__
    __graft_entry__.build()
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "netflix": run_netflix(args, dev)}
    print(json.dumps(res["netflix"]), file=sys.stderr, flush=True)
    if not args.skip_density:
        res["density"] = run_density(args, dev)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
