#!/usr/bin/env python
"""Headline benchmark: BNMF Gibbs + VB update sweeps on synthetic 65536 x 32768 fp64, 20 % missing, K=20
(BASELINE.json config 4).  One JSON line on stdout; see DESIGN.md section "Measurement".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows I --cols J --K K]
                    [--workload sweep|cv|small|nmtf] [--dump-outputs DIR]

A "step" is one Gibbs sweep plus one VB sweep (all U columns, all V columns, tau, train metrics each);
value = sweeps per second over both.  N>1 (torchrun): rows of R / R^T are sharded across ranks
(bnmtf_b200/parallel.py) -- strong scaling of the same matrix.

Besides the timing the line carries a PARITY block: the GPU classes and the CPU checker (the reference's own classes
from baseline/_ref when that copy exists, else the oracle port) run the same 4096 x 2048, K=20 problem from the same
seeded 'random' start, and the largest relative differences of factors, MSE, ELBO and tau are printed.  The CPU side
of that run is also the cpu_baseline sample.

--workload cv / small: the replica decomposition (independent fits, one per GPU); --workload nmtf: the tri-factorisation
at the headline shape -- see bench_replicas.py.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HBM_FALLBACK_GBS = 6650.0
# ncu dram bytes (read + write) per launch at the full 65536 x 32768 shape on one GPU, by digit count
# (profiles/r01d_ncu_summary.txt, re-measured in profiles/r02_ncu_summary.txt); scaled by 1/world for a shard
RX_TRAFFIC_PER_ENTRY = {7: 15.15e9 / 2.0 ** 31, 6: 12.97e9 / 2.0 ** 31}
GRAM_TRAFFIC_PER_LAUNCH = {7: 1.6e9, 6: 1.25e9}
TRAFFIC_SOURCE = ("ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per launch at the full shape on one GPU, taken inside "
                  "the sweep (profiles/r03_k_gram_umma_details.txt: 1.05 GB + 0.20 GB; profiles/r03_k_rx_umma_details.txt: "
                  "12.93 GB + 0.04 GB), not re-measured in this run")
FP64_PEAK_TFLOPS = 37.1   # measured here: tools/microbench/fp64_pipes.cu -> profiles/r01_microbench_fp64_pipes.txt
DTYPE = "f64 (statistics: 48-bit fixed point, exact int8 tcgen05 accumulation; solver, moments, draws: IEEE fp64)"
PRIORS = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
PARITY_SHAPE = (4096, 2048)
PARITY_TOL = 1e-9


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------------
def make_synthetic(I, J, K, device, seed=0, row_lo=0, row_hi=None, tile=4096):
    """SURVEY.md 8(d): U0,V0 ~ Exp(1) (numpy RandomState(seed)), R = U0 V0^T + N(0,1), M = rand >= 0.2, generated in
    row tiles directly into the library's device layout (rows [row_lo,row_hi) only).  torch is the data generator
    here -- this is input synthesis, outside every timed region."""
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream, ld_for
    rng = np.random.RandomState(seed)
    U0 = rng.exponential(1.0, size=(I, K))
    V0 = rng.exponential(1.0, size=(J, K))
    row_hi = I if row_hi is None else row_hi
    n = row_hi - row_lo
    ld = ld_for(J)
    R = torch.zeros((n, ld), dtype=torch.float64, device=device)
    bits = torch.zeros((n, ld // 32), dtype=torch.int32, device=device)
    V0d = torch.from_numpy(V0).to(device)
    n_obs = 0
    for t0 in range(0, n, tile):
        t1 = min(n, t0 + tile)
        g = torch.Generator(device=device)
        g.manual_seed(seed * 1000003 + (row_lo + t0))       # tile-keyed: identical data for any sharding
        U0d = torch.from_numpy(U0[row_lo + t0:row_lo + t1]).to(device)
        Rt = U0d @ V0d.T + torch.randn((t1 - t0, J), dtype=torch.float64, device=device, generator=g)
        Mt = (torch.rand((t1 - t0, J), dtype=torch.float64, device=device, generator=g) >= 0.2).to(torch.float64)
        n_obs += float(Mt.sum())
        _lib.call("bnmtf_pack_dataset_f64", _ptr(Rt), _ptr(Mt), t1 - t0, J, ld, R[t0:].data_ptr(), bits[t0:].data_ptr(), _stream())
        torch.cuda.synchronize()
        del Rt, Mt
    return R, bits, n_obs


def build_roofline(engs, prof, I, J, K, n_obs, sweep_s, world=1):
    """Roofline block of the JSON line (DESIGN.md section 5).  The dominant kernel of a sweep is the per-row Gram
    (tcgen05 int8 tensor pipe); the R-streaming kernel is reported beside it against the HBM roof.  world > 1: the
    per-launch figures are per rank (1/world of the entries), the whole-sweep HBM figure is against world x peak."""
    hbm_peak, hbm_kind = measured_peaks()
    N = float(I) * J / world
    n_obs = n_obs / world
    e0 = next(iter(engs.values()))
    # the Gram kernel is timed inside a long, power-capped run: the sustained cuBLAS figure is its denominator
    # (B200_PROFILING.md); the burst figure is reported beside it
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            pk = json.load(fh)
        bf16, bf16_burst = float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])), float(pk["bf16_tflops"])
        bf16_kind = "measured, sustained"
    except Exception:
        bf16, bf16_burst, bf16_kind = 1400.0, 1590.0, "fallback, sustained"
    b_alg_sweep = 2.0 * N * world * 8.125
    out = {"kernel_ms": prof,
           "sweep_hbm": {"algorithmic_bytes_per_sweep": b_alg_sweep, "achieved_gbs": b_alg_sweep / sweep_s / 1e9,
                         "peak_gbs": hbm_peak * world, "peak_kind": hbm_kind,
                         "frac": b_alg_sweep / sweep_s / 1e9 / (hbm_peak * world)}}
    from bnmtf_b200 import _lib
    digits = _lib.call("bnmtf_fixed_point_digits")       # bytes per fixed-point image (6 by default)
    out["fixed_point_digits"] = digits
    if e0.gram == "umma":
        # exact fixed-point Gram: 0/1 selection matrix (rows x cols) times the int8 digit slices of K(K+1)/2 (+K
        # variance, VB) (+K column-sum, metrics phase) product columns; algorithmic ops = 2 * rows * cols * digit columns
        ops, ach = {}, {}
        for k, e in engs.items():
            nc = K * (K + 1) // 2 + (K if e.vb else 0)
            ops[k] = 2.0 * N * (nc + 0.5 * (K if e.metrics_mode == "stats" else 0)) * digits
            ach[k] = ops[k] / (prof[k]["stats_gram"] * 1e-3) / 1e12
        mean_ach = sum(ach.values()) / len(ach)
        peak = 2.0 * bf16
        out.update({"bound": "tensor", "kernel": "k_gram_umma (tcgen05.mma kind::i8, TMEM accumulators, TMA-fed)",
                    "achieved": mean_ach, "peak": peak, "unit": "TFLOP/s", "frac": mean_ach / peak,
                    "traffic": (GRAM_TRAFFIC_PER_LAUNCH.get(digits) / world if GRAM_TRAFFIC_PER_LAUNCH.get(digits) else None),
                    "peak_source": "2 x bf16_tflops_sustained of MEASURED_PEAKS.json (%s): the int8 tensor rate of B200 is "
                                   "twice the bf16 rate; ops are int8 multiply-adds x 2; the kernel is timed inside the "
                                   "power-capped sweep loop" % bf16_kind,
                    "frac_of_burst_peak": mean_ach / (2.0 * bf16_burst),
                    "traffic_source": TRAFFIC_SOURCE,
                    "per_mode_achieved_tops": ach})
    else:
        miss = N - n_obs
        pairs = K * (K + 1) / 2.0
        fl = {"gibbs": miss * (pairs + K) * 2.0, "vb": miss * (pairs + 2 * K) * 2.0}
        ach = {k: fl[k] / (prof[k]["stats_gram"] * 1e-3) / 1e12 for k in engs}
        mean_ach = sum(ach.values()) / len(ach)
        out.update({"bound": "tensor", "kernel": "k_stats_gram (fp64 DMMA, mma.sync.m8n8k4.f64)", "achieved": mean_ach,
                    "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": mean_ach / FP64_PEAK_TFLOPS, "traffic": None,
                    "peak_source": "fp64 DMMA peak measured by tools/microbench/fp64_pipes.cu"})
    # the HBM-bound kernel: streams R once per phase (`digits` digit-plane bytes per entry for the tcgen05 kernel,
    # 8 + 1/8 bytes for the fp64 kernel).  Two durations: alone on all SMs, and inside the sweep, where it runs on
    # `split` SMs beside the Gram kernel
    bpe = float(digits) if e0.rx == "umma" else 8.125
    rx_ms = sum(prof[k]["stats_rx"] for k in engs) / len(engs)
    rx_in = sum(prof[k].get("stats_rx_in_sweep", 0.0) for k in engs) / len(engs)
    rx_gbs = N * bpe / (rx_ms * 1e-3) / 1e9
    hk = {"bound": "hbm", "kernel": "k_rx_umma (tcgen05 digit planes)" if e0.rx == "umma" else "k_stats_rx (fp64 DMMA)",
          "achieved": rx_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": rx_gbs / hbm_peak,
          "duration": "timed alone on all SMs",
          "algorithmic_bytes_per_launch": N * bpe, "peak_kind": hbm_kind + " (copy bandwidth)",
          "traffic": RX_TRAFFIC_PER_ENTRY.get(digits, 0) * N if (e0.rx == "umma" and digits in RX_TRAFFIC_PER_ENTRY) else None,
          "traffic_source": TRAFFIC_SOURCE}
    if rx_in > 0:
        hk["in_sweep"] = {"ms": rx_in, "achieved": N * bpe / (rx_in * 1e-3) / 1e9,
                          "frac": N * bpe / (rx_in * 1e-3) / 1e9 / hbm_peak,
                          "note": "same kernel inside the sweep: %d SMs, the Gram kernel on the others" % e0.split}
    out["hbm_kernel"] = hk
    return out


# ------------------------------------------------------------------------------------------------------
# CPU side: the reference's own classes (baseline/_ref, made by __graft_entry__.build() from /root/reference with
# oracle/ref_shim.py) or, when that copy is absent, the oracle port.  Test/measurement infrastructure only.
# ------------------------------------------------------------------------------------------------------
def load_reference():
    if not os.path.isdir(os.path.join(REF_DIR, "BNMTF", "code", "models")):
        return None
    try:
        from oracle import ref_shim
        return ref_shim.load(REF_DIR)
    except Exception as exc:                                   # a broken copy must not take the benchmark down
        sys.stderr.write("bench: baseline/_ref present but not importable (%s: %s); using the oracle port\n" % (type(exc).__name__, exc))
        return None


def quiet():
    return contextlib.redirect_stdout(io.StringIO())


def sample_problem(I, J, K, seed=0):
    rng = np.random.RandomState(seed)
    U0, V0 = rng.exponential(1.0, size=(I, K)), rng.exponential(1.0, size=(J, K))
    R = U0 @ V0.T + rng.normal(size=(I, J))
    M = (rng.rand(I, J) >= 0.2).astype(float)
    return R, M


def blas_threads():
    try:
        import threadpoolctl
        info = threadpoolctl.threadpool_info()
        return max(i.get("num_threads", 1) for i in info) if info else 1
    except Exception:
        return os.cpu_count() or 1


class CpuTimer:
    """Wall and process-CPU seconds of a region: cpu/wall = the number of cores the region really kept busy."""

    def __init__(self):
        self.wall = self.cpu = 0.0

    def __enter__(self):
        self._w, self._c = time.time(), time.process_time()
        return self

    def __exit__(self, *a):
        self.wall += time.time() - self._w
        self.cpu += time.process_time() - self._c


class CpuModels:
    """The three BNMF models of the CPU side behind one interface (reference classes or oracle port)."""

    def __init__(self, R, M, K, ref):
        self.R, self.M, self.K, self.ref = R, M, K, ref
        self.kind = "reference" if ref is not None else "port"

    # Each start_* seeds numpy exactly like gpu_parity_run() does before the GPU class's initialise('random').
    def start_vb(self, seed):
        np.random.seed(seed)
        if self.ref is not None:
            m = self.ref.bnmf_vb_optimised(self.R, self.M, self.K, PRIORS)
            with quiet():
                m.initialise("random")
            return m
        from oracle import bnmtf_oracle as orc
        o = orc.OracleBNMF(self.R, self.M, self.K, PRIORS, mode="vb")
        muU = np.random.exponential(scale=1.0 / o.lambdaU)
        muV = np.random.exponential(scale=1.0 / o.lambdaV)
        o.init_vb(muU, muV)
        return o

    def sweep_vb(self, m):
        if self.ref is not None:
            with quiet():
                m.run(1)
            return {"MSE": m.all_performances["MSE"][-1]}
        return m.sweep()

    def state_vb(self, m):
        if self.ref is not None:
            return {"expU": m.expU, "expV": m.expV, "varU": m.varU, "varV": m.varV, "exptau": m.exptau, "elbo": m.elbo()}
        return {"expU": m.U, "expV": m.V, "varU": m.varU, "varV": m.varV, "exptau": m.exptau, "elbo": m.elbo()}

    def start_point(self, seed, mode):
        """Gibbs / ICM model at a seeded 'random' start."""
        np.random.seed(seed)
        if self.ref is not None:
            m = (self.ref.bnmf_gibbs_optimised if mode == "gibbs" else self.ref.nmf_icm)(self.R, self.M, self.K, PRIORS)
            with quiet():
                m.initialise("random")
            return m
        from oracle import bnmtf_oracle as orc
        o = orc.OracleBNMF(self.R, self.M, self.K, PRIORS, mode=mode)
        U = np.random.exponential(scale=1.0 / o.lambdaU)
        V = np.random.exponential(scale=1.0 / o.lambdaV)
        o.set_state(U, V)
        return o

    def conditionals(self, m, k):
        if self.ref is not None:
            tU = np.asarray(m.tauU(k), dtype=float)
            tV = np.asarray(m.tauV(k), dtype=float)
            return {"tauU": tU, "muU": np.asarray(m.muU(tU, k), dtype=float), "tauV": tV, "muV": np.asarray(m.muV(tV, k), dtype=float)}
        tU, mU = m.column_params(k, "U")
        tV, mV = m.column_params(k, "V")
        return {"tauU": tU, "muU": mU, "tauV": tV, "muV": mV}

    def sweep_point(self, m, mode):
        if self.ref is not None:
            with quiet():
                m.run(1) if mode == "gibbs" else m.run(1, minimum_TN=0.0)
            return {"MSE": m.all_performances["MSE"][-1]}
        return m.sweep()


def cpu_side(K, shape=PARITY_SHAPE, vb_sweeps=2, icm_sweeps=2, want_parity=True):
    """Run the CPU checker on the parity problem; its timed VB and Gibbs sweeps are the cpu_baseline sample."""
    I, J = shape
    R, M = sample_problem(I, J, K)
    cpu = CpuModels(R, M, K, load_reference())
    res = {"kind": cpu.kind, "shape": shape}
    t_vb, t_g = CpuTimer(), CpuTimer()
    m = cpu.start_vb(11)
    res["vb"] = []
    for _ in range(vb_sweeps if want_parity else 1):
        with t_vb:
            perf = cpu.sweep_vb(m)
        st = cpu.state_vb(m)
        st = {k: (np.array(v, dtype=float).copy() if isinstance(v, np.ndarray) else float(v)) for k, v in st.items()}
        st["MSE"] = float(perf["MSE"])
        res["vb"].append(st)
    res["vb_sweeps_timed"] = len(res["vb"])
    g = cpu.start_point(12, "gibbs")
    if want_parity:
        res["gibbs_cond"] = cpu.conditionals(g, K // 2)
    with t_g:
        cpu.sweep_point(g, "gibbs")
    if want_parity:
        c = cpu.start_point(13, "icm")
        res["icm"] = []
        for _ in range(icm_sweeps):
            perf = cpu.sweep_point(c, "icm")
            res["icm"].append({"U": np.array(c.U, dtype=float).copy(), "V": np.array(c.V, dtype=float).copy(),
                               "tau": float(c.tau), "MSE": float(perf["MSE"])})
    res["s_vb"], res["s_gibbs"] = t_vb.wall / res["vb_sweeps_timed"], t_g.wall
    res["cores_busy"] = (t_vb.cpu + t_g.cpu) / max(1e-9, t_vb.wall + t_g.wall)
    res["cpu_seconds"] = t_vb.wall + t_g.wall
    return res


def gpu_parity_run(K, distributed, shape=PARITY_SHAPE, vb_sweeps=2, icm_sweeps=2):
    """The GPU classes on the parity problem from the same seeded 'random' starts (every rank when sharded)."""
    import bnmtf_b200
    I, J = shape
    R, M = sample_problem(I, J, K)
    kw = {"distributed": True} if distributed else {}
    out = {"vb": [], "icm": []}
    np.random.seed(11)
    m = bnmtf_b200.bnmf_vb_optimised(R, M, K, PRIORS, seed=5, **kw)
    m.initialise("random")
    for _ in range(vb_sweeps):
        m.run(1)
        out["vb"].append({"expU": m.expU.copy(), "expV": m.expV.copy(), "varU": m.varU.copy(), "varV": m.varV.copy(),
                          "exptau": float(m.exptau), "elbo": float(m.all_elbo[-1]), "MSE": float(m.all_performances["MSE"][-1])})
    # the device's TN variance against the reference's formula (truncated_normal_vector.py:62-73) at the device's own mu, tau
    from oracle import bnmtf_oracle as orc
    out["var_same_inputs"] = max(rel_err(m.varU, orc.tn_variance(m.muU, m.tauU)), rel_err(m.varV, orc.tn_variance(m.muV, m.tauV)))
    np.random.seed(12)
    g = bnmtf_b200.bnmf_gibbs_optimised(R, M, K, PRIORS, seed=6, **kw)
    g.initialise("random")
    k = K // 2
    tU, tV = g.tauU(k), g.tauV(k)
    out["gibbs_cond"] = {"tauU": tU, "muU": g.muU(tU, k), "tauV": tV, "muV": g.muV(tV, k)}
    np.random.seed(13)
    c = bnmtf_b200.nmf_icm(R, M, K, PRIORS, seed=7, **kw)
    c.initialise("random")
    for _ in range(icm_sweeps):
        c.run(1, minimum_TN=0.0)
        out["icm"].append({"U": c.U.copy(), "V": c.V.copy(), "tau": float(c.tau), "MSE": float(c.all_performances["MSE"][-1])})
    del m, g, c
    return out


def rel_err(a, b):
    """max |a - b| / (|b| + 0.01 max|b|): relative, with entries near zero measured against 1 % of the largest."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = float(np.abs(b).max()) if b.size else 0.0
    if scale == 0.0:
        return float(np.abs(a - b).max()) if a.size else 0.0
    return float(np.max(np.abs(a - b) / (np.abs(b) + 0.01 * scale)))


def parity_block(gpu, cpu, K, world):
    I, J = cpu["shape"]
    blk = {"problem": "%dx%d, K=%d, 20%% missing, seeded 'random' starts; same kernels as the headline run "
                      "(tcgen05 Gram + R.X, SM split, CUDA graph%s)" % (I, J, K, ", %d-way sharded" % world if world > 1 else ""),
           "checker": "reference classes (baseline/_ref)" if cpu["kind"] == "reference" else "oracle port (oracle/bnmtf_oracle.py)",
           "measure": "max |gpu - cpu| / (|cpu| + 0.01 max|cpu|)", "tolerance": PARITY_TOL}
    worst = 0.0
    vb = {"sweeps": len(cpu["vb"]), "max_rel_factors": 0.0, "max_rel_variances": 0.0, "max_rel_mse": 0.0, "max_rel_elbo": 0.0,
          "max_rel_exptau": 0.0}
    elbo_finite = 0
    for a, b in zip(gpu["vb"], cpu["vb"]):
        vb["max_rel_factors"] = max(vb["max_rel_factors"], rel_err(a["expU"], b["expU"]), rel_err(a["expV"], b["expV"]))
        vb["max_rel_variances"] = max(vb["max_rel_variances"], rel_err(a["varU"], b["varU"]), rel_err(a["varV"], b["varV"]))
        vb["max_rel_mse"] = max(vb["max_rel_mse"], abs(a["MSE"] / b["MSE"] - 1.0))
        if np.isfinite(a["elbo"]) and np.isfinite(b["elbo"]):
            vb["max_rel_elbo"] = max(vb["max_rel_elbo"], abs(a["elbo"] / b["elbo"] - 1.0))
            elbo_finite += 1
        elif not (a["elbo"] == b["elbo"] or (np.isnan(a["elbo"]) and np.isnan(b["elbo"]))):
            vb["max_rel_elbo"] = float("inf")          # one side finite, the other not
        vb["max_rel_exptau"] = max(vb["max_rel_exptau"], abs(a["exptau"] / b["exptau"] - 1.0))
    vb["elbo_finite_sweeps"] = elbo_finite   # log(erfc) underflows to -inf on both sides while entries sit > 38 sigma below 0
    vb["variance_note"] = ("the reference's TN variance sigma^2 (1 - lambda (lambda - x)) is evaluated from exp(-x*x/2) and "
                           "erfc(x/sqrt2), whose argument roundings differ: for strongly truncated entries its value depends "
                           "on the last bits of x with amplitude ~1e-13 x^4 (x = -mu sqrt(tau) up to 30), so two evaluations "
                           "whose mu differ by 1e-10 differ by that much; max_rel_variances_same_inputs is the device value "
                           "against the same formula in numpy at the DEVICE's own mu, tau")
    if "var_same_inputs" in gpu:
        vb["max_rel_variances_same_inputs"] = gpu["var_same_inputs"]
    blk["vb"] = vb
    worst = max(worst, *[v for k, v in vb.items() if k.startswith("max_") and k != "max_rel_variances"])
    icm = {"sweeps": len(cpu["icm"]), "max_rel_factors": 0.0, "max_rel_mse": 0.0, "max_rel_tau": 0.0}
    for a, b in zip(gpu["icm"], cpu["icm"]):
        icm["max_rel_factors"] = max(icm["max_rel_factors"], rel_err(a["U"], b["U"]), rel_err(a["V"], b["V"]))
        icm["max_rel_mse"] = max(icm["max_rel_mse"], abs(a["MSE"] / b["MSE"] - 1.0))
        icm["max_rel_tau"] = max(icm["max_rel_tau"], abs(a["tau"] / b["tau"] - 1.0))
    blk["icm"] = icm
    worst = max(worst, *[v for k, v in icm.items() if k.startswith("max_")])
    gc = {"column": K // 2}
    for name in ("tauU", "muU", "tauV", "muV"):
        gc["max_rel_" + name] = rel_err(gpu["gibbs_cond"][name], cpu["gibbs_cond"][name])
        worst = max(worst, gc["max_rel_" + name])
    blk["gibbs_conditionals"] = gc
    blk["worst"] = worst
    blk["pass"] = bool(worst <= PARITY_TOL)
    blk["pass_covers"] = "factors, MSE, ELBO, tau, conditionals, variances at the same inputs (trajectory variances: see variance_note)"
    return blk


# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own classes (baseline/_ref; the oracle port if that copy is missing) on the
    host cores.  A step = one Gibbs + one VB sweep, as in our arm, on a bounded sample of the workload: the largest
    rung of 512x256 ... 4096x2048 for which warmup + steps fit about 150 s; value = sweeps/s at the full shape by linear
    extrapolation in I*J (the reference needs ~6 dense I x J temporaries per column update: the full shape does not
    fit host RAM and would take ~45 minutes per sweep)."""
    I, J, K = args.rows, args.cols, args.K
    t_start = time.time()
    ref = load_reference()
    n_steps = args.warmup + args.steps
    per_entry_step = 2.8e-6                                    # s per matrix entry per (Gibbs + VB) step, K=20, measured here
    rung = (256, 128)
    for cand in ((512, 256), (1024, 512), (2048, 1024), (4096, 2048)):
        if cand[0] * cand[1] * per_entry_step * (K / 20.0) * n_steps <= 150.0:
            rung = cand
    Is, Js = min(rung[0], I), min(rung[1], J)
    R, M = sample_problem(Is, Js, K)
    cpu = CpuModels(R, M, K, ref)
    vb = cpu.start_vb(11)
    gb = cpu.start_point(12, "gibbs")
    for _ in range(args.warmup):
        cpu.sweep_point(gb, "gibbs"), cpu.sweep_vb(vb)
    tm = CpuTimer()
    with tm:
        for _ in range(args.steps):
            cpu.sweep_point(gb, "gibbs"), cpu.sweep_vb(vb)
    step_s = tm.wall / max(1, args.steps)
    scale = (float(I) * J) / (float(Is) * Js)
    value = 2.0 / (step_s * scale)
    cores_busy = tm.cpu / max(1e-9, tm.wall)
    sample = ("%d steps of one Gibbs + one VB sweep of the %s at %dx%d, K=%d (%.1f s); sweeps/s at %dx%d by linear extrapolation "
              "in I*J" % (args.steps, "reference's bnmf_gibbs_optimised / bnmf_vb_optimised (baseline/_ref)" if ref is not None
                          else "oracle port", Is, Js, K, tm.wall, I, J))
    line = {"impl": "reference", "metric": "BNMF Gibbs+VB sweeps/sec at %dx%d K=%d" % (I, J, K), "value": value,
            "unit": "sweeps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BNMF Gibbs+VB sweep, %dx%d fp64, 20%% missing, K=%d" % (I, J, K),
                       "sample_shape": [Is, Js], "extrapolation_factor": scale,
                       "note": "ms_per_step is the measured time of one step on the sample; value is extrapolated to the full "
                               "shape, which does not fit host RAM in the reference's formulation"},
            "cpu_baseline": {"value": value, "unit": "sweeps/s", "cores": max(1, int(round(cores_busy))), "kind": cpu.kind,
                             "sample": sample, "cores_busy_measured": cores_busy, "blas_threads": blas_threads(),
                             "host_cores": os.cpu_count()},
            "e2e": {"value": value, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.time() - t_start}
    print(json.dumps(line))


def checksum(models, engs):
    """State after a fixed number of sweeps from the same seeded start: identical for every sharding of the same
    problem (Gibbs: bit for bit, the Philox counters are keyed by global row; VB: to rounding)."""
    import torch
    from bnmtf_b200 import engine
    out = {}
    for k, e in engs.items():
        sc = e.scalars.cpu().numpy()
        out[k] = {"sweeps": int(e.sweeps_done), "sum_U": float(e.U.fac[:e.U.n].sum().item()),
                  "sum_V": float(e.V.fac[:e.V.n].sum().item()), "sum_U2": float((e.U.fac[:e.U.n] ** 2).sum().item()),
                  "tau": float(sc[engine.S_TAU]), "train_MSE": float(sc[engine.S_MSE])}
    torch.cuda.synchronize()
    return out


DUMP_BYTES = 64 * 10 ** 6        # 64 MB, decimal


def dump_outputs(engs, steps, out_dir, rank):
    """What the timed sweeps handed back, as run(steps) would give it to a caller, written to out_dir/<name>.npy (float64):
    gibbs_U / gibbs_V, vb_{exp,var,mu,tau}{U,V} (the classes' attribute names) and <mode>_trace, one row per timed sweep
    of tau, MSE, R^2, Rp (all_tau / all_exp_tau and all_performances).  The VB ELBO (all_elbo) is left out: from this
    seeded random start it is -inf, as in the reference, while strongly truncated entries make log erfc underflow
    (DESIGN.md section 5, parity; at the headline shape through at least the first 23 sweeps,
    profiles/r04_dump_repeat.txt), so it holds nothing to compare.  Beyond DUMP_BYTES the factor arrays keep a fixed seeded
    sample of their rows, the same rows for every array of a side; rows_U.npy / rows_V.npy then hold the row indices."""
    import torch
    if "vb" in engs:
        engs["vb"].gather_params()          # mu / tau of the other ranks' rows (no-op on one GPU)
    torch.cuda.synchronize()
    if rank != 0:
        return
    sides = ([], [])                        # (name, device tensor [n, K]) per factor side
    small = {}
    for mode, e in engs.items():
        for side, (f, s) in enumerate(((e.U, "U"), (e.V, "V"))):
            fields = ((f.fac, "exp"), (f.var, "var"), (f.mu, "mu"), (f.tauf, "tau")) if e.vb else ((f.fac, ""),)
            for t, attr in fields:
                sides[side].append(("%s_%s%s" % (mode, attr, s), t[:f.n]))
        last = e.sweeps_done - e.trace_base
        small[mode + "_trace"] = e.trace[last - steps:last, :4].cpu().numpy()     # tau, MSE, R^2, Rp
    n = [sides[i][0][1].shape[0] for i in (0, 1)]
    row_bytes = [sum(t[0].numel() * 8 for _, t in sides[i]) for i in (0, 1)]
    room = DUMP_BYTES - sum(a.nbytes for a in small.values()) - 4096
    frac = min(1.0, room / float(sum(n[i] * (row_bytes[i] + 8) for i in (0, 1))))
    out = dict(small)
    for i, s in enumerate("UV"):
        idx = None
        if frac < 1.0:
            idx = np.sort(np.random.RandomState(i).choice(n[i], int(n[i] * frac), replace=False))
            out["rows_" + s] = idx.astype(np.float64)
            idx = torch.from_numpy(idx).to(sides[i][0][1].device)
        for name, t in sides[i]:
            out[name] = (t if idx is None else t.index_select(0, idx)).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="sweep", choices=["sweep", "cv", "small", "nmtf"])
    ap.add_argument("--rows", type=int, default=65536)
    ap.add_argument("--cols", type=int, default=32768)
    ap.add_argument("--K", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--sustained-s", type=float, default=2.5)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state left by the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "sweep" or args.impl != "ours"):
        ap.error("--dump-outputs needs --workload sweep --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload != "sweep":
        import bench_replicas
        return bench_replicas.main(args, rank, world)
    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return

    import torch
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from bnmtf_b200 import _lib, bnmf, engine
    I, J, K = args.rows, args.cols, args.K
    dist = None
    if world > 1:
        import torch.distributed as dist
        from bnmtf_b200 import parallel
        parallel.init_process_group("nccl")
        R, bits, RT, bitsT, n_obs = parallel.make_synthetic_shards(I, J, K, device, rank, world)
        ds = engine.Dataset.from_device(R, bits, I, J, RT, bitsT, n_obs=n_obs, world=world, rank=rank)
    else:
        R, bits, n_obs = make_synthetic(I, J, K, device)
        ds = engine.Dataset.from_device(R, bits, I, J, n_obs=n_obs)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    # seeded 'random' start (numpy seeds 1, 2: the same host draws on every rank and for every world size)
    models = {}
    for i, (mode, cls) in enumerate((("gibbs", bnmf.bnmf_gibbs_optimised), ("vb", bnmf.bnmf_vb_optimised))):
        m = cls.from_dataset(ds, K, PRIORS, seed=1)
        np.random.seed(1 + i)
        m.initialise("random")
        models[mode] = m
    engs = {k: m._engine() for k, m in models.items()}
    for m in models.values():
        m._push()
    # ---- device-resident timing: state stays in HBM, K sweeps of each sampler back to back -------------------
    for e in engs.values():
        e.alloc_trace(args.warmup + args.steps + 64)
    for _ in range(args.warmup):
        for e in engs.values():
            e.sweep()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in engs}
    launches0 = _lib.launch_count[0]
    t_all0 = torch.cuda.Event(enable_timing=True)
    t_all1 = torch.cuda.Event(enable_timing=True)
    t_all0.record()
    for k, e in engs.items():
        ev[k][0].record()
        for _ in range(args.steps):
            e.sweep()
        ev[k][1].record()
    t_all1.record()
    barrier()
    launches = _lib.launch_count[0] - launches0
    times = torch.tensor([t_all0.elapsed_time(t_all1)] + [ev[k][0].elapsed_time(ev[k][1]) for k in ("gibbs", "vb")],
                         dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    total_ms, g_ms, v_ms = (float(x) for x in times.cpu())
    value = 2.0 * args.steps / (total_ms / 1e3)
    state = checksum(models, engs)                     # after exactly warmup + steps sweeps, for every N
    if args.dump_outputs:
        dump_outputs(engs, args.steps, args.dump_outputs, rank)

    # ---- sustained figure: the same loop for >= sustained_s seconds (the board settles at its power cap) ----------
    sustained = None
    if args.sustained_s > 0:
        n_sus = max(args.steps, int(args.sustained_s / max(1e-4, total_ms / 1e3 / (2.0 * args.steps)) / 2.0) + 1)
        for e in engs.values():
            e.alloc_trace(n_sus + 8)
        for e in engs.values():
            e.sweep()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for e in engs.values():
            for _ in range(n_sus):
                e.sweep()
        s1.record()
        barrier()
        st = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=device)
        if dist is not None:
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
        sustained = {"sweeps_per_s": 2.0 * n_sus / (float(st.item()) / 1e3), "seconds": float(st.item()) / 1e3, "sweeps": 2 * n_sus}

    # ---- per-kernel timings for the roofline block -----------------------------------------------------------
    prof = {k: e.profile_sweep(reps=2 if world == 1 else 1) for k, e in engs.items()}
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- end to end through the public class API: host state in, host state out, every step -------------------
    e2e = None
    if not args.no_e2e:
        for m in models.values():
            m.run(1)
        barrier()
        t0 = time.time()
        for m in models.values():
            for _ in range(args.steps):
                m.run(1)
        barrier()
        dt = torch.tensor([time.time() - t0], dtype=torch.float64, device=device)
        if dist is not None:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = sum(m._xfer_bytes()[0] for m in models.values()) / 2.0
        d2h = sum(m._xfer_bytes()[1] for m in models.values()) / 2.0
        e2e = {"value": 2.0 * args.steps / float(dt.item()), "unit": "sweeps/s", "h2d_bytes_per_step": int(h2d * world),
               "d2h_bytes_per_step": int(d2h * world),
               "note": "model.run(1) per step through the class API: factor state DMA'd from the model's page-locked host "
                       "arrays, one sweep, state + trace read back into them; bytes are summed over ranks (each rank moves "
                       "only its own rows of the factor state; the fused peer exchange replicates them); R itself "
                       "(16 GiB) is resident like a dataset"}

    # ---- parity at the benchmark's kernel configuration (every rank runs the GPU side; rank 0 the CPU side) ------
    gpu_par = None
    if not args.no_parity:
        for m in models.values():
            m._eng = None
        del models, engs, ds, R, bits
        if world > 1:
            del RT, bitsT
        torch.cuda.empty_cache()
        gpu_par = gpu_parity_run(K, distributed=world > 1)
    if dist is not None:
        barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    # ---- roofline ------------------------------------------------------------------------------------------------
    N = float(I) * J
    sweep_s = total_ms / 1e3 / (2.0 * args.steps)
    roofline = build_roofline_from(prof, I, J, K, n_obs, sweep_s, world)
    par_txt = ("rows of R and of R^T sharded over %d ranks; each updated factor row is stored into every peer's copy by the "
               "solver kernel itself (NVLink P2P stores into symmetric memory, one cross-GPU barrier per phase); one "
               "24-double all-reduce per sweep (NCCL)" % world) if world > 1 else "single GPU"
    line = {"metric": "BNMF Gibbs+VB sweeps/sec at %dx%d K=%d" % (I, J, K), "value": value, "unit": "sweeps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / (2.0 * args.steps),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": "BNMF Gibbs+VB sweep, %dx%d fp64, 20%% missing, K=%d" % (I, J, K),
                       "parallelism": par_txt, "init": "seeded 'random' start (numpy seeds 1, 2)",
                       "l2": "inputs (2 x %.1f GiB of digit planes per sweep) far larger than L2" % (N * 6 / 2 ** 30),
                       "gibbs_sweeps_per_s": args.steps / (g_ms / 1e3), "vb_sweeps_per_s": args.steps / (v_ms / 1e3),
                       "sustained": sustained, "state_after_timed_region": state, "observed_fraction": n_obs / N},
            "roofline": roofline, "e2e": e2e, "gpu_launches": launches, "clocks": sampler.summary()}
    if not (args.no_cpu_baseline and args.no_parity):
        cpu = cpu_side(K, want_parity=not args.no_parity)
        s_g, s_v = cpu["s_gibbs"] * N / (PARITY_SHAPE[0] * PARITY_SHAPE[1]), cpu["s_vb"] * N / (PARITY_SHAPE[0] * PARITY_SHAPE[1])
        line["cpu_baseline"] = {"value": 2.0 / (s_g + s_v), "unit": "sweeps/s", "cores": max(1, int(round(cpu["cores_busy"]))),
                                "kind": cpu["kind"],
                                "sample": "%d VB + 1 Gibbs sweep of the %s at %dx%d, K=%d (%.1f s of CPU work); sweeps/s at the "
                                          "full shape by linear extrapolation in I*J -- the full shape needs >62 GB in the "
                                          "reference's formulation" % (cpu["vb_sweeps_timed"],
                                                                      "reference's own classes (baseline/_ref)" if cpu["kind"] == "reference" else "oracle port",
                                                                      PARITY_SHAPE[0], PARITY_SHAPE[1], K, cpu["cpu_seconds"]),
                                "cores_busy_measured": cpu["cores_busy"], "blas_threads": blas_threads(), "host_cores": os.cpu_count(),
                                "seconds_per_sweep_sample": {"gibbs": cpu["s_gibbs"], "vb": cpu["s_vb"]}}
        if gpu_par is not None:
            line["parity"] = parity_block(gpu_par, cpu, K, world)
    print(json.dumps(line))


def build_roofline_from(prof, I, J, K, n_obs, sweep_s, world):
    """build_roofline() needs only a few engine attributes: carried in prof['_meta'] so that the engines themselves can
    be freed before the parity run."""
    class E:
        pass
    engs = {}
    for k, p in prof.items():
        e = E()
        e.gram, e.rx, e.vb, e.metrics_mode, e.split = p["_meta"]["gram"], p["_meta"]["rx"], k == "vb", p["_meta"]["metrics_mode"], p["_meta"]["split"]
        engs[k] = e
    prof = {k: {n: v for n, v in p.items() if n != "_meta"} for k, p in prof.items()}
    return build_roofline(engs, prof, I, J, K, n_obs, sweep_s, world)


if __name__ == "__main__":
    main()
