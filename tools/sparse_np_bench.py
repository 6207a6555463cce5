"""Sparse input of the non-probabilistic models (NMF, NMTF multiplicative updates) on one B200: sweeps/s at the Netflix
shape, the CUDA-event time of every call of a sweep and the S-phase share, the achieved bytes/s of the row update, the
device memory high-water mark, and the observed fraction at which the dense NP path overtakes the sparse one.

    python tools/sparse_np_bench.py [--out profiles/r08_sparse_np_bench.json] [--iterations 30] [--percents 0.5 1 2 5 10 20]

The matrix is tools/sparse_bench.py's netflix_like() (480 189 x 17 770, 100 480 507 observed entries) with its values
raised to at least 0.01, so that r log(r/p) (the I-divergence) is finite.  Sweeps/s come from the CUDA events run()
records per iteration (replayed as a CUDA graph), over the iterations after the capture.  Per-call times come from three
eager iterations with a pair of CUDA events around every library call.  Prints one JSON line, and writes it to --out.
"""
import argparse
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STEP = {"bnmtf_csr_np_row_update_f64": "row_update", "bnmtf_csr_np_s_update_f64": "S_phase",
        "bnmtf_csr_np_metrics_f64": "metrics", "bnmtf_small_matmul_f64": "small_matmul"}


def _sparse_bench():
    spec = importlib.util.spec_from_file_location("sparse_bench", os.path.join(ROOT, "tools", "sparse_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def sweeps_per_s(model, iterations):
    model.run(iterations)
    t = model.all_times
    return (len(t) - 3) / (t[-1] - t[2])


def call_times(model, reps=3):
    """ms per sweep of every step and of every call, from `reps` eager iterations with events around each call."""
    import torch
    from bnmtf_b200 import _lib
    real = _lib.call
    rec = []

    def timed(name, *args):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = real(name, *args)
        e1.record()
        rec.append((name, e0, e1))
        return r
    _lib.call = timed
    try:
        model.run(reps)                     # fewer than 8 iterations: no CUDA graph
        torch.cuda.synchronize()
    finally:
        _lib.call = real
    steps, calls = {}, {}
    for name, a, b in rec:
        ms = a.elapsed_time(b)
        steps[STEP.get(name, name)] = steps.get(STEP.get(name, name), 0.0) + ms / reps
        calls.setdefault(name, []).append(ms)
    # calls_ms: ms of each call of one sweep, averaged over the reps sweeps
    out = {"steps_ms": steps, "total_ms": sum(steps.values()),
           "calls_ms": {k: [round(float(np.mean(v[i::len(v) // reps])), 4) for i in range(len(v) // reps)]
                        for k, v in calls.items()}}
    out["S_phase_share"] = steps.get("S_phase", 0.0) / out["total_ms"]
    return out


def row_update_bytes(nnz, rows, cols, K):
    """Bytes one row-update phase must move, counted from shapes: the CSR streams (int32 column, fp64 value per entry), the
    phase's factor read and written once (rows x K), and each entry's row of the other factor gathered once (nnz x K)."""
    return {"csr": 12 * nnz, "factor_rw": 16 * rows * K, "gather": 8 * nnz * K,
            "hbm_min": 12 * nnz + 16 * rows * K + 8 * cols * K}


def run_netflix(args, dev, sb, res):
    import torch
    from bnmtf_b200 import NMF, NMTF, data
    R = sb.netflix_like(seed=args.seed, device=dev)
    R.data = np.maximum(R.data, 0.01)
    torch.cuda.reset_peak_memory_stats(dev)
    ds = data.upload_sparse(R, device=dev)
    I, J, nnz = R.shape[0], R.shape[1], int(R.nnz)
    res.update({"shape": [I, J], "nnz": nnz, "device_csr_GB": ds.nbytes() / 1e9})
    runs = [("NMF", 20, None)] + [("NMTF", kl, kl) for kl in args.KL]
    for name, K, L in runs:
        np.random.seed(1)
        m = NMF.from_dataset(ds, K) if L is None else NMTF.from_dataset(ds, K, L)
        m.initialise()
        rate = sweeps_per_s(m, args.iterations)
        r = {"K": K, "L": L, "sweeps_per_s": rate, "sweep_ms": 1e3 / rate, "calls": call_times(m),
             "final_MSE": m.all_performances["MSE"][-1], "final_I_div": m.all_i_div[-1]}
        ru = r["calls"]["calls_ms"].get("bnmtf_csr_np_row_update_f64", [])
        if len(ru) >= 2:
            rows_cols = ((I, J, K), (J, I, K)) if L is None else ((I, J, K), (J, I, L))
            r["row_update"] = []
            for (rows, cols, w), ms in zip(rows_cols, ru[-2:]):
                b = row_update_bytes(nnz, rows, cols, w)
                r["row_update"].append({"ms": ms, "bytes": b, "hbm_min_GB_per_s": b["hbm_min"] / ms / 1e6,
                                        "csr_plus_gather_GB_per_s": (b["csr"] + b["gather"]) / ms / 1e6})
        if L is not None:
            r["S_phase_bytes_min_per_pass"] = 28 * nnz
            sms = r["calls"]["steps_ms"].get("S_phase", 0.0)
            r["S_phase_GB_per_s_at_28B"] = 28 * nnz * K * L / sms / 1e6 if sms else None
        res["%s_K%d" % (name, K) + ("" if L is None else "_L%d" % L)] = r
        print(json.dumps({name: r}), file=sys.stderr, flush=True)
        del m
    res["peak_device_GB"] = torch.cuda.max_memory_allocated(dev) / 1e9
    del ds
    torch.cuda.empty_cache()


def run_density(args, dev, sb):
    """NMF (K = 20) sweeps/s of the sparse and the dense path on the same seeded 65536 x 32768 matrix at each fraction."""
    import torch
    from bnmtf_b200 import NMF, data, engine
    I, J, K = 65536, 32768, 20
    out = []
    for pct in args.percents:
        nnz = int(round(pct / 100.0 * I * J))
        R = sb.make_sparse(I, J, nnz, seed=args.seed + 7, device=dev, uniform=True)
        R.data = np.maximum(R.data, 0.01)
        row = {"percent": pct, "nnz": nnz}
        ds = data.upload_sparse(R, device=dev)
        np.random.seed(1)
        m = NMF.from_dataset(ds, K)
        m.initialise()
        row["sparse_sweeps_per_s"] = sweeps_per_s(m, args.iterations)
        sp_idiv = m.all_i_div[-1]
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
        m = NMF.from_dataset(dd, K)
        m.initialise()
        row["dense_sweeps_per_s"] = sweeps_per_s(m, args.iterations)
        row["I_div_rel_diff"] = abs(m.all_i_div[-1] / sp_idiv - 1)
        del m, dd, Rd, bits
        torch.cuda.empty_cache()
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    faster = [r["percent"] for r in out if r["dense_sweeps_per_s"] > r["sparse_sweeps_per_s"]]
    return {"shape": [I, J], "K": K, "rows": out, "dense_faster_from_percent": min(faster) if faster else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--KL", type=int, nargs="+", default=[10, 20])
    ap.add_argument("--iterations", type=int, default=30)
    ap.add_argument("--percents", type=float, nargs="*", default=[0.5, 1, 2, 5, 10, 20])
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    import torch
    sb = _sparse_bench()
    dev = torch.device("cuda", 0)
    res = {"gpu": sb.gpu_info()}
    run_netflix(args, dev, sb, res)
    if args.percents:
        res["density"] = run_density(args, dev, sb)
    res["power_state_after"] = sb.gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
