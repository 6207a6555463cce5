#!/usr/bin/env python
"""Sweep the SM split of the two statistics kernels (BNMTF_SPLIT: SMs given to the R.X kernel, the Gram kernel's CTA
pairs take the rest) over the flagship benchmark.  Each point is one `bench.py --no-parity --no-cpu-baseline --no-e2e`
subprocess; the passes over the split values alternate so that drift of the clocks hits every value alike.

    python tools/split_sweep.py --K 20 --splits 48,56,64,72,80 --passes 2 --out sweep_K20.json

Prints one line per run and a table (median over the passes) and writes every JSON line to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(K, split, args):
    env = dict(os.environ, BNMTF_SPLIT=str(split))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--K", str(K), "--steps", str(args.steps),
           "--warmup", str(args.warmup), "--sustained-s", str(args.sustained_s), "--no-parity", "--no-cpu-baseline",
           "--no-e2e"]
    out = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=args.timeout)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if out.returncode or not lines:
        raise RuntimeError("bench.py failed (K=%d, split=%d):\n%s" % (K, split, out.stderr[-3000:]))
    return json.loads(lines[-1])


def summary(line):
    c, km = line["config"], line["roofline"]["kernel_ms"]
    return {"value": line["value"], "gibbs": c["gibbs_sweeps_per_s"], "vb": c["vb_sweeps_per_s"],
            "sustained": (c["sustained"] or {}).get("sweeps_per_s"),
            "rx_in_sweep": [km[m]["stats_rx_in_sweep"] for m in ("gibbs", "vb")],
            "gram_in_sweep": [km[m]["stats_gram_in_sweep"] for m in ("gibbs", "vb")],
            "sm_mhz": line["clocks"].get("sm_mhz"), "reasons": line["clocks"].get("reasons")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=20)
    ap.add_argument("--splits", default="48,56,64,72,80")
    ap.add_argument("--passes", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sustained-s", type=float, default=2.5)
    ap.add_argument("--timeout", type=float, default=600)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    splits = [int(s) for s in args.splits.split(",")]
    if any(s <= 0 or s % 2 for s in splits):
        ap.error("split values must be positive and even (the Gram kernel runs as CTA pairs)")
    runs = []
    for p in range(args.passes):
        for s in (splits if p % 2 == 0 else splits[::-1]):
            line = run(args.K, s, args)
            runs.append({"K": args.K, "split": s, "pass": p, "summary": summary(line), "line": line})
            print(json.dumps({"K": args.K, "split": s, "pass": p, **runs[-1]["summary"]}), flush=True)
    with open(args.out, "w") as f:
        for r in runs:
            f.write(json.dumps(r) + "\n")
    print("K=%d   split   sweeps/s (median)   gibbs    vb    sustained   R.X / Gram in sweep, Gibbs (ms)" % args.K)
    for s in splits:
        rs = [r["summary"] for r in runs if r["split"] == s]
        med = lambda key: statistics.median(x[key] for x in rs)
        sus = [x["sustained"] for x in rs if x["sustained"]]
        print("        %4d   %7.2f  [%s]   %6.2f  %6.2f   %s   %.2f / %.2f" % (
            s, med("value"), " ".join("%.2f" % x["value"] for x in rs), med("gibbs"), med("vb"),
            "%6.2f" % statistics.median(sus) if sus else "   -  ",
            statistics.median(x["rx_in_sweep"][0] for x in rs), statistics.median(x["gram_in_sweep"][0] for x in rs)))


if __name__ == "__main__":
    main()
