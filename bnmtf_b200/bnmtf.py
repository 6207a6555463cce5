"""Drop-in classes for the reference's tri-factorisation models R ~ F S G^T, backed by the B200 engine.

    bnmtf_gibbs_optimised  (code/models/bnmtf_gibbs_optimised.py:55)
    bnmtf_vb_optimised     (code/models/bnmtf_vb_optimised.py:59)
    nmtf_icm               (code/models/nmtf_icm.py:49)

Same constructor arguments, method names, return values, attribute names and assertion messages as the reference.
All arithmetic of the update sweep runs in CUDA kernels (csrc/stats.cu for the two streaming passes over R per
sweep, csrc/nmtf.cu + csrc/solve.cu for the F / S / G updates on the row statistics).
"""
import itertools
import math
import os
import random

import numpy as np
import scipy.sparse
import torch

from . import _lib
from .data import training_csr, validate_sparse
from .bnmf import METRICS, QUALITY, _TwoFactorBase, _elbo_alpha_s_correction, _metrics_from_sums
from .engine import (CSR_METRIC_CTAS, MODE, Dataset, Factor, Partition, SparseDataset, capture_graph, thread_flags, S_BETA_S, S_ELBO,
                     S_ESD, S_LOGTAU, S_TAU, _ptr, _stream, gram_len, kp_for, require_cuda)


class BNMTFEngine:
    """Device state and sweep driver for one (R, M, K, L)."""

    def __init__(self, dataset, K, L, mode, alpha, beta, seed=0):
        self._alloc(dataset, K, L, mode, alpha, beta, seed)
        ds, dev = dataset, dataset.device
        I, J = ds.I, ds.J
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
        self.nseg_m = max(1, min(ds.ldJ // 128, -(-1776 // ((I + 127) // 128))))
        self.mpart = f64(((I + 127) // 128) * self.nseg_m * 8)
        # Statistics kernels: the fp64 mma.sync ones at toy / GDSC sizes (latency-bound there, fewer launches), the tcgen05
        # fixed-point ones of the two-factor engine for large matrices (BNMTF_NMTF_STATS=umma|dmma overrides).  A dataset
        # with outlier rows (Dataset.wide) keeps fp64; the per-phase dynamic-range guard of the two-factor engine is not
        # wired into the tri-factor kernels.
        want = os.environ.get("BNMTF_NMTF_STATS", "umma" if I * J >= (1 << 22) else "dmma")
        self.stats_impl = "dmma"
        if want == "umma" and max(self.K, self.L) <= 32:
            for side in (0, 1):
                ds.ensure_planes(side)
            if not any(ds.wide.values()):
                self.stats_impl = "umma"
                self.wsrx_bytes = max(_lib.call("bnmtf_rx_umma_workspace_bytes", d, ld) for d, ld in ((self.L, ds.ldJ), (self.K, ds.ldI)))
                self.wsrx = torch.zeros(self.wsrx_bytes + 1024, dtype=torch.uint8, device=dev)
                self.wsrx_ptr = (self.wsrx.data_ptr() + 1023) // 1024 * 1024
                self.ws_bytes = max(_lib.call("bnmtf_gram_umma_workspace_bytes", d, int(self.vb), ld)
                                    for d, ld in ((self.L, ds.ldJ), (self.K, ds.ldI)))
                self.ws = torch.zeros(self.ws_bytes + 1024, dtype=torch.uint8, device=dev)
                self.ws_ptr = (self.ws.data_ptr() + 1023) // 1024 * 1024
        # training metrics of a sweep: "stats" = from the column statistics of the G phase (csrc/nmtf.cu::k_nmtf_mstat: no
        # third pass over R; the direct pass runs only when the device-side cancellation guard trips, as in the two-factor
        # engine), "direct" = always the pass over R
        self.metrics_mode = os.environ.get("BNMTF_METRICS", "stats" if self.stats_impl == "umma" else "direct")
        self.statics = f64(3)
        _lib.call("bnmtf_masked_metrics_f64", _ptr(ds.R), _ptr(ds.bits), I, ds.ldJ, _ptr(self.FS.Xp), _ptr(self.G.Xp),
                  self.L, self.nseg_m, 0, _ptr(self.mpart), _ptr(self.m8), 0, _stream())
        self.statics.copy_(self.m8[4:7])
        if ds.n_obs is None:
            ds.n_obs = float(self.statics[2].item())
        self.polarity = 0 if ds.n_obs >= 0.5 * I * J else 1
        self._set_omega()

    def _alloc(self, dataset, K, L, mode, alpha, beta, seed):
        """Factors, S, the statistics records of both phases and the scratch of the sweep: what every format needs."""
        self.ds, self.K, self.L, self.mode = dataset, int(K), int(L), mode
        self.m, self.vb = MODE[mode], mode == "vb"
        self.alpha, self.beta, self.seed = float(alpha), float(beta), int(seed) & (2 ** 64 - 1)
        ds, dev = dataset, dataset.device
        I, J, D = ds.I, ds.J, self.K * self.L
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
        self.F = Factor(Partition(I), self.K, dev, self.vb)
        self.G = Factor(Partition(J), self.L, dev, self.vb)
        self.FS = Factor(Partition(I), self.L, dev, False)          # F S, for the prediction metrics
        self.S = {k: f64(self.K, self.L) for k in ("fac", "var", "mu", "tauf", "lam")}
        self.S["lam"].fill_(1.0)
        self.scalars = f64(16)
        self.iter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.iter_scratch = torch.zeros(1, dtype=torch.int64, device=dev)
        # static device buffers for the per-sweep update orders (VB: the reference's shuffles) and the CUDA graph of a sweep:
        # at these sizes a sweep is ~30 launches of a few microseconds each, i.e. bound by launch latency when issued eagerly
        self.order_buf = {"S": torch.zeros(max(1, D), dtype=torch.int32, device=dev),
                          "F": torch.zeros(self.K, dtype=torch.int32, device=dev),
                          "G": torch.zeros(self.L, dtype=torch.int32, device=dev)}
        self.use_graph = int(os.environ.get("BNMTF_GRAPH", "1")) >= 1
        self._graph = self._graph_key = self._graph_seen = None
        self._graph_kernels = 0
        self.trace, self.trace_cap, self.trace_base, self.sweeps_done = None, 0, 0, 0
        KPk, KPl, GLk, GLl = kp_for(self.K), kp_for(self.L), gram_len(self.K), gram_len(self.L)
        # statistics of the rows of R w.r.t. G (dimension L) and of the rows of R^T w.r.t. F (dimension K)
        self.row = {"RX": f64(I, KPl), "G": f64(I, GLl), "SV": f64(I, KPl), "full": f64(GLl + KPl)}
        self.col = {"RX": f64(J, KPk), "G": f64(J, GLk), "SV": f64(J, KPk), "full": f64(GLk + KPk)}
        n, KPm, GLm = max(I, J), max(KPk, KPl), max(GLk, GLl)
        self.eff = {"RX": f64(n, KPm), "G": f64(n, GLm), "SV": f64(n, KPm)}      # effective-factor statistics
        self.gscratch = f64(296 * (GLm + KPm))       # bnmtf_gram_full_f64: up to 296 partial results
        self.nparts = int(_lib.call("bnmtf_nmtf_sq_parts", I, self.K, self.L, int(self.vb)))    # row partitions of the S-phase reduction
        self.sq_len = D * D + 2 * D
        self.sq_part = f64(self.nparts * int(_lib.call("bnmtf_nmtf_sq_scratch_len", self.K, self.L, int(self.vb))))
        self.sq_out = f64(self.sq_len)
        self.extra = f64(J)
        self.red = f64(24)
        self.m8, self.el8, self.ex1 = self.red[0:8], self.red[8:16], self.red[16:17]
        self.nb_terms = 32 if max(I * self.K, J * self.L) <= (1 << 16) else 296      # CTAs of the ELBO factor terms
        self.elpart = f64(3 * self.nb_terms * 8)
        self.guard = 1e-5
        self.mstat, self.mstat_part, self.sums4, self.m8d = f64(J, 4), f64(256), f64(4), f64(8)
        self.flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self._side = self._ev = None
        self.sterm = None

    def _set_omega(self):
        from scipy.special import gammaln, psi
        self.size_Omega = float(self.ds.n_obs)
        self.alpha_s = self.alpha + self.size_Omega / 2.0
        self.digamma_alpha_s, self.lgamma_alpha = float(psi(self.alpha_s)), float(gammaln(self.alpha))
        self.lgamma_alpha_s = float(gammaln(self.alpha_s))

    # ---- small problems: the whole run as ONE kernel (csrc/small.cu::k_small_tri) -------------------------------
    def small_cluster(self):
        if getattr(self, "_small_c", None) is None:
            ok = os.environ.get("BNMTF_SMALL", "1") != "0"
            self._small_c = int(_lib.call("bnmtf_small_tri_cluster_size", self.ds.I, self.ds.J, self.K, self.L, int(self.vb))) if ok else 0
            if self._small_c:
                import ctypes
                D, dev = self.K * self.L, self.ds.device
                self._small_partial = torch.zeros(16 * 16 + 32, dtype=torch.float64, device=dev)
                self._small_H = torch.zeros(17 * (D * D + 2 * D), dtype=torch.float64, device=dev)
                tab = lambda *ts: (ctypes.c_void_p * 5)(*[_ptr(t) or None for t in ts])
                S = self.S
                self._small_tabs = (tab(self.F.fac, self.F.var, self.F.mu, self.F.tauf, self.F.lam),
                                    tab(self.G.fac, self.G.var, self.G.mu, self.G.tauf, self.G.lam),
                                    tab(S["fac"], S["var"] if self.vb else None, S["mu"], S["tauf"], S["lam"]))
        return self._small_c

    def sweep_many(self, sweeps, minimum_TN=0.0, samples=None, times=None, sums=None, orders=None):
        """`sweeps` iterations of run() in one launch.  samples = (all_F, all_S, all_G): device tensors for the Gibbs draw of
        every sweep; orders: int32 device tensor [sweeps, K*L + K + L] (VB: the three shuffled orders of every sweep)."""
        assert sums is None
        import ctypes
        ds, D = self.ds, self.K * self.L
        trace_ptr = _ptr(self.trace) - self.trace_base * 64 if self.trace is not None else 0
        aF, aS, aG = samples if samples is not None else (None, None, None)
        HL = D * D + 2 * D
        tF, tG, tS = self._small_tabs
        _lib.call("bnmtf_small_tri_sweeps_f64", self.m, _ptr(ds.R), _ptr(ds.bits), _ptr(ds.RT), _ptr(ds.bitsT), ds.I, ds.J, ds.ldJ,
                  ds.ldI, self.K, self.L, ctypes.cast(tF, ctypes.c_void_p), ctypes.cast(tG, ctypes.c_void_p),
                  ctypes.cast(tS, ctypes.c_void_p), _ptr(self.scalars), trace_ptr, _ptr(self.iter), self.trace_base + self.trace_cap,
                  self.alpha, self.beta, self.digamma_alpha_s, self.lgamma_alpha, self.lgamma_alpha_s, float(minimum_TN), self.seed,
                  int(sweeps), _ptr(orders), _ptr(aF), _ptr(aS), _ptr(aG), _ptr(self._small_partial), _ptr(self._small_H),
                  self._small_H.data_ptr() + 8 * 16 * HL, _ptr(times), _stream())
        self.sweeps_done += int(sweeps)

    # ---- layer 1 ------------------------------------------------------------------------------------------
    @staticmethod
    def split(dim):
        if "BNMTF_SPLIT" in os.environ:
            return int(os.environ["BNMTF_SPLIT"])
        return 64 if dim > 16 else (80 if dim > 8 else 96)

    def _stats(self, st, R, bits, rows, ld, other, dim, need_rx=True):
        other.pad()
        if self.polarity == 0:
            _lib.call("bnmtf_gram_full_f64", _ptr(other.Xp), _ptr(other.Vp), other.n, dim, ld, _ptr(st["full"]),
                      _ptr(self.gscratch), _stream())
        if self.stats_impl == "umma":
            # the two-factor model's tcgen05 kernels (exact fixed-point int8 GEMMs, csrc/rx_umma.cu, csrc/gram_umma.cu): the
            # statistics of the tri-factorisation ARE two-factor statistics w.r.t. G (rows) and F (columns); one segment,
            # because the transform / S-reduction kernels read one record per row
            side = 0 if R is self.ds.R else 1
            sums = 1 if (side == 1 and self.metrics_mode == "stats") else 0        # slot (k, K): masked column sums of F

            def rx(max_ctas):
                planes, rscale = self.ds.ensure_planes(side)[:2]
                _lib.call("bnmtf_stats_rx_umma_f64", planes.data_ptr(), _ptr(rscale), _ptr(R), _ptr(bits), rows, ld, other.n,
                          _ptr(other.Xp), dim, 1, max_ctas, _ptr(st["RX"]), self.wsrx_ptr, self.wsrx_bytes, _stream())

            def gram():
                _lib.call("bnmtf_stats_gram_umma_f64", _ptr(bits), rows, ld, other.n, _ptr(other.Xp), _ptr(other.Vp), dim,
                          self.polarity, 1, 128 if ld >= 256 else 64, 1, sums, 0, _ptr(st["G"]), _ptr(st["SV"]) if self.vb else 0,
                          self.ws_ptr, self.ws_bytes, _stream())
            split = self.split(dim)
            if need_rx and split > 0:
                # SM split of the two-factor engine (engine.py::_stats_kernels): the HBM-bound R.X kernel on `split` SMs of
                # a high-priority stream, the tensor-bound Gram kernel on the rest
                if self._side is None:
                    self._side = torch.cuda.Stream(device=self.ds.device, priority=-1)
                    self._ev = [torch.cuda.Event(), torch.cuda.Event()]
                main = torch.cuda.current_stream()
                self._ev[0].record(main)
                self._side.wait_event(self._ev[0])
                with torch.cuda.stream(self._side):
                    rx(split)
                    self._ev[1].record(self._side)
                gram()
                main.wait_event(self._ev[1])
            else:
                if need_rx:
                    rx(0)
                gram()
            return
        if need_rx:
            _lib.call("bnmtf_stats_rx_f64", _ptr(R), _ptr(bits), rows, ld, _ptr(other.Xp), dim, 1, _ptr(st["RX"]), _stream())
        _lib.call("bnmtf_stats_gram_f64", _ptr(bits), rows, ld, _ptr(other.Xp), _ptr(other.Vp), dim, self.polarity, 1,
                  _ptr(st["G"]), _ptr(st["SV"]) if self.vb else 0, _stream())

    def stats_rows(self, need_rx=True):
        ds = self.ds
        self._stats(self.row, ds.R, ds.bits, ds.I, ds.ldJ, self.G, self.L, need_rx)

    def stats_cols(self, need_rx=True):
        ds = self.ds
        self._stats(self.col, ds.RT, ds.bitsT, ds.J, ds.ldI, self.F, self.K, need_rx)

    # ---- layer 2 ------------------------------------------------------------------------------------------
    def _order(self, order):
        """order: None (natural order), a list of indices, or ("static", name): the engine's own buffer, filled by sweep()."""
        if order is None:
            return 0, None
        if isinstance(order, tuple) and order[0] == "static":
            t = self.order_buf[order[1]]
            return _ptr(t), t
        t = torch.tensor([int(x) for x in order], dtype=torch.int32, device=self.ds.device)
        return _ptr(t), t

    def _outer(self, me, st, rows, Ks, Lo, Smat, varS, order, n_order, apply, minimum_TN, salt, want_sterm, use_iter):
        _lib.call("bnmtf_nmtf_transform_f64", rows, Ks, Lo, self.polarity, 1 if self.vb else 0, _ptr(st["RX"]), _ptr(st["G"]),
                  _ptr(st["SV"]) if self.vb else 0, _ptr(st["full"]), _ptr(Smat), _ptr(varS) if self.vb else 0,
                  _ptr(self.eff["RX"]), _ptr(self.eff["G"]), _ptr(self.eff["SV"]) if self.vb else 0, _stream())
        optr, keep = self._order(order)
        if order is not None:
            n_order = Ks if isinstance(order, tuple) else len(order)
        elif n_order is None:
            n_order = Ks
        if want_sterm:
            self.sterm = torch.zeros((rows, Ks), dtype=torch.float64, device=self.ds.device)
        _lib.call("bnmf_row_solve_f64", self.m, rows, Ks, 1, 1, 1, _ptr(self.eff["RX"]), _ptr(self.eff["G"]),
                  _ptr(self.eff["SV"]) if self.vb else 0, 0, _ptr(me.fac), _ptr(me.var), _ptr(me.mu), _ptr(me.tauf),
                  _ptr(me.lam), _ptr(self.scalars), optr, n_order, 1 if apply else 0, float(minimum_TN), self.seed,
                  _ptr(self.iter if use_iter else self.iter_scratch), salt, 0,
                  _ptr(self.sterm) if want_sterm else 0, 0, 0, 0, 0, 0, 0, 0, _stream())
        del keep

    def phase_F(self, order=None, n_order=None, apply=True, minimum_TN=0.0, want_sterm=False, use_iter=True):
        self._outer(self.F, self.row, self.ds.I, self.K, self.L, self.S["fac"], self.S["var"], order, n_order, apply,
                    minimum_TN, 0, want_sterm, use_iter)

    def phase_G(self, order=None, n_order=None, apply=True, minimum_TN=0.0, want_sterm=False, use_iter=True):
        ST = self.S["fac"].T.contiguous()
        vST = self.S["var"].T.contiguous()
        self._outer(self.G, self.col, self.ds.J, self.L, self.K, ST, vST, order, n_order, apply, minimum_TN, 1, want_sterm,
                    use_iter)

    def phase_S(self, order=None, apply=True, minimum_TN=0.0, use_iter=True):
        """order: flat indices k*L + l (None: all, row-major as itertools.product(range(K), range(L)))."""
        D = self.K * self.L
        _lib.call("bnmtf_nmtf_sq_f64", self.ds.I, self.K, self.L, self.polarity, 1 if self.vb else 0, _ptr(self.row["RX"]),
                  _ptr(self.row["G"]), _ptr(self.row["SV"]) if self.vb else 0, _ptr(self.row["full"]), _ptr(self.F.fac),
                  _ptr(self.F.var) if self.vb else 0, _ptr(self.sq_part), self.nparts, _ptr(self.sq_out), _stream())
        optr, keep = self._order(order)
        n_order = D if (order is None or isinstance(order, tuple)) else len(order)
        S = self.S
        base = self.sq_out.data_ptr()
        _lib.call("bnmtf_coord_solve_f64", self.m, D, base, base + 8 * D * D, base + 8 * (D * D + D), _ptr(S["lam"]),
                  _ptr(S["fac"]), _ptr(S["var"]) if self.vb else 0, _ptr(S["mu"]), _ptr(S["tauf"]), _ptr(self.scalars),
                  optr, n_order, 1 if apply else 0, float(minimum_TN), self.seed,
                  _ptr(self.iter if use_iter else self.iter_scratch), 2, _stream())
        del keep

    def metrics(self, bits=None, gated=False):
        """Masked sums over `bits` (default: the training mask) with the current factors -> self.m8.  gated: -> self.m8d,
        and the pass over R only runs if the device flag of the statistics-based metrics is raised."""
        ds = self.ds
        _lib.call("bnmtf_small_matmul_f64", _ptr(self.F.fac), _ptr(self.S["fac"]), ds.I, self.K, self.L, 0,
                  _ptr(self.FS.fac), _stream())
        self.FS.pad()
        self.G.pad()
        bits = ds.bits if bits is None else bits
        statics = _ptr(self.statics) if bits is ds.bits else 0
        _lib.call("bnmtf_masked_metrics_f64", _ptr(ds.R), _ptr(bits), ds.I, ds.ldJ, _ptr(self.FS.Xp), _ptr(self.G.Xp),
                  self.L, self.nseg_m, statics, _ptr(self.mpart), _ptr(self.m8d if gated else self.m8),
                  _ptr(self.flag) if gated else 0, _stream())

    def metrics_from_stats(self):
        """Training metrics right after the G phase of a sweep: the column statistics are current w.r.t. F, and S and G
        are the new ones, so the three masked sums follow from them column by column (k_nmtf_mstat)."""
        ds = self.ds
        _lib.call("bnmtf_nmtf_mstat_f64", ds.J, self.K, self.L, self.polarity, _ptr(self.col["RX"]), _ptr(self.col["G"]),
                  _ptr(self.col["full"]), _ptr(self.G.fac), _ptr(self.S["fac"]), _ptr(self.mstat), _stream())
        _lib.call("bnmtf_mstat_reduce_f64", _ptr(self.mstat), ds.J, _ptr(self.mstat_part), _ptr(self.sums4), _stream())
        _lib.call("bnmtf_metrics_from_sums_f64", _ptr(self.sums4), _ptr(self.statics), self.guard, _ptr(self.m8),
                  _ptr(self.flag), _stream())
        self.metrics(gated=True)                 # returns at once unless the guard tripped
        _lib.call("bnmtf_select_metrics_f64", _ptr(self.flag), _ptr(self.m8d), _ptr(self.m8), _stream())

    def vb_extra(self):
        """Variance terms of exp_square_diff; the column statistics must be current w.r.t. F."""
        S = self.S
        _lib.call("bnmtf_nmtf_extra_f64", self.ds.J, self.K, self.L, self.polarity, _ptr(self.col["G"]), _ptr(self.col["SV"]),
                  _ptr(self.col["full"]), _ptr(self.G.fac), _ptr(self.G.var), _ptr(S["fac"]), _ptr(S["var"]),
                  _ptr(self.extra), _stream())
        _lib.call("bnmtf_reduce1_f64", _ptr(self.extra), self.ds.J, _ptr(self.ex1), _stream())

    def vb_terms(self):
        nb = self.nb_terms
        S = self.S
        triples = ((self.F.fac, self.F.var, self.F.mu, self.F.tauf, self.F.lam, self.ds.I * self.K),
                   (S["fac"], S["var"], S["mu"], S["tauf"], S["lam"], self.K * self.L),
                   (self.G.fac, self.G.var, self.G.mu, self.G.tauf, self.G.lam, self.ds.J * self.L))
        for i, (e, v, m, t, l, n) in enumerate(triples):
            _lib.call("bnmtf_vb_factor_terms_f64", _ptr(e), _ptr(v), _ptr(m), _ptr(t), _ptr(l), n,
                      self.elpart[i * nb * 8:].data_ptr(), nb, _stream())
        _lib.call("bnmtf_reduce8_f64", _ptr(self.elpart), 3 * nb, _ptr(self.el8), _stream())

    def finish(self, update_tau=True, record=True):
        trace_ptr = _ptr(self.trace) - self.trace_base * 64 if (record and self.trace is not None) else 0
        nfe = self.ds.I * self.K + self.K * self.L + self.ds.J * self.L
        _lib.call("bnmf_finish_sweep_f64", self.m, self.alpha, self.beta, self.digamma_alpha_s, self.lgamma_alpha,
                  self.lgamma_alpha_s, nfe, _ptr(self.m8), _ptr(self.ex1), _ptr(self.el8), _ptr(self.scalars), trace_ptr,
                  _ptr(self.iter if record else self.iter_scratch), self.trace_base + self.trace_cap if record else 0,
                  self.seed, 1 if update_tau else 0, 0, _stream())
        if record:
            self.sweeps_done += 1

    def refresh_scalars(self, update_tau=True):
        self.red.zero_()
        if self.vb:
            self.stats_cols(need_rx=False)
            self.vb_extra()
            self.vb_terms()
        self.metrics()
        self.finish(update_tau=update_tau, record=False)

    def sweep(self, minimum_TN=0.0, order=None):
        """One iteration of run().  Gibbs / ICM: F, S, G (bnmtf_gibbs_optimised.py:152-166).  VB: S, F, G in the
        host-supplied (shuffled) orders (bnmtf_vb_optimised.py:171-190).  The orders go into static device buffers, so the
        launch sequence has fixed arguments and is replayed as a CUDA graph from the third sweep of a run on."""
        static = None
        if self.vb and order is not None and all(order.get(k) is not None for k in "SFG"):
            for k in "SFG":
                # pageable source: the runtime stages the bytes before returning, so the host may run sweeps ahead of the device
                self.order_buf[k].copy_(torch.tensor([int(x) for x in order[k]], dtype=torch.int32))
            static = {k: ("static", k) for k in "SFG"}
            order = None
        if self.use_graph and order is None and not getattr(thread_flags, "no_graph", False):
            key = (self.trace.data_ptr() if self.trace is not None else 0, self.trace_base, self.trace_cap, float(minimum_TN),
                   static is not None)
            if self._graph is not None and self._graph_key == key:
                self._graph.replay()
                _lib.launch_count[0] += self._graph_kernels
                self.sweeps_done += 1
                return
            if self._graph_seen == key and self.trace_cap >= 8:       # (a short run does not repay the capture)
                done, count0 = self.sweeps_done, _lib.launch_count[0]
                g = capture_graph(lambda: self._sweep_eager(minimum_TN, static))          # captured, not executed
                self._graph_kernels = _lib.launch_count[0] - count0
                _lib.launch_count[0] = count0
                self.sweeps_done = done
                self._graph, self._graph_key = g, key
                g.replay()
                _lib.launch_count[0] += self._graph_kernels
                self.sweeps_done += 1
                return
            self._graph_seen = key
        self._sweep_eager(minimum_TN, static if static is not None else order)

    def _sweep_eager(self, minimum_TN=0.0, order=None):
        if self.vb:
            oS, oF, oG = (order or {}).get("S"), (order or {}).get("F"), (order or {}).get("G")
            self.stats_rows()
            self.phase_S(oS)
            self.phase_F(oF)
            self.stats_cols()
            self.phase_G(oG)
            self.vb_extra()
            self.vb_terms()
        else:
            self.stats_rows()
            self.phase_F(minimum_TN=minimum_TN)
            self.phase_S(minimum_TN=minimum_TN)
            self.stats_cols()
            self.phase_G(minimum_TN=minimum_TN)
        if self.metrics_mode == "stats":
            self.metrics_from_stats()
        else:
            self.metrics()
        self.finish(update_tau=True, record=True)

    def alloc_trace(self, iterations):
        self.trace_cap = int(iterations)
        self.trace = torch.zeros((max(1, self.trace_cap), 8), dtype=torch.float64, device=self.ds.device)
        self.trace_base = self.sweeps_done


class SparseBNMTFEngine(BNMTFEngine):
    """BNMTFEngine on a SparseDataset.  The format decision lives here: the statistics of a phase come from one
    bnmtf_csr_stats_f64 call over the phase's CSR (rows of R against G, rows of R^T against F; fp64, polarity 1, one
    record per row: no digit planes, no unmasked totals), the sweep's metrics from the column statistics with
    bnmtf_csr_metrics_f64 as the gated direct pass.  Transform, S-phase reduction, solvers, end of the sweep and CUDA-graph
    replay are BNMTFEngine's, which read the same records at polarity 1."""

    def __init__(self, dataset, K, L, mode, alpha, beta, seed=0):
        if dataset.world != 1:
            raise ValueError("sparse input runs on one GPU")
        self._alloc(dataset, K, L, mode, alpha, beta, seed)
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dataset.device)
        KPm, GLm = max(kp_for(self.K), kp_for(self.L)), max(gram_len(self.K), gram_len(self.L))
        smax = max(1, dataset.csr[0].n_slots, dataset.csr[1].n_slots)
        # chunk partials of the long rows, for the wider of the two phases
        self.RXc, self.Gc = f64(smax, KPm), f64(smax, GLm)
        self.SVc = f64(smax, KPm) if self.vb else None
        self.mpart = f64(CSR_METRIC_CTAS * 8)
        self.stats_impl, self.metrics_mode, self.polarity = "csr", "stats", 1
        self._small_c = 0               # never the single-kernel small path
        self.statics = dataset.statics.clone()
        self._set_omega()

    def _csr_stats(self, side, st, other, need_rx):
        c = self.ds.csr[side]
        other.pad()
        _lib.call("bnmtf_csr_stats_f64", _ptr(c.rowptr), _ptr(c.colidx), _ptr(c.val), _ptr(c.item_begin), _ptr(c.item_row),
                  _ptr(c.item_slot), c.n_items, c.chunk, _ptr(c.heavy_row), _ptr(c.heavy_first), c.n_heavy, _ptr(other.Xp),
                  _ptr(other.Vp), other.K, _ptr(st["RX"]) if need_rx else 0, _ptr(st["G"]), _ptr(st["SV"]) if self.vb else 0,
                  _ptr(self.RXc), _ptr(self.Gc), _ptr(self.SVc), _stream())

    def stats_rows(self, need_rx=True):
        self._csr_stats(0, self.row, self.G, need_rx)

    def stats_cols(self, need_rx=True):
        self._csr_stats(1, self.col, self.F, need_rx)

    def metrics(self, bits=None, gated=False):
        """The seven sums over the entry set `bits` (None: the training entries; else a DeviceCSR from pack_mask) with the
        prediction (F S) G^T -> self.m8 (gated: -> self.m8d, only if the device flag is raised)."""
        _lib.call("bnmtf_small_matmul_f64", _ptr(self.F.fac), _ptr(self.S["fac"]), self.ds.I, self.K, self.L, 0,
                  _ptr(self.FS.fac), _stream())
        self.FS.pad()
        self.G.pad()
        entries = self.ds.csr[0] if bits is None else bits
        entries.metrics(self.FS.Xp, self.G.Xp, self.L, self.mpart, self.m8d if gated else self.m8,
                        self.flag if gated else None)

    def small_cluster(self):
        return 0


def tri_engine_for(dataset, K, L, mode, alpha, beta, seed=0):
    """The engine that runs on `dataset`: SparseBNMTFEngine for a SparseDataset, BNMTFEngine otherwise."""
    cls = SparseBNMTFEngine if isinstance(dataset, SparseDataset) else BNMTFEngine
    return cls(dataset, K, L, mode, alpha, beta, seed=seed)


# =====================================================================================================
class _ThreeFactorBase(object):
    _mode = None
    compute_MSE, compute_R2, compute_Rp = _TwoFactorBase.compute_MSE, _TwoFactorBase.compute_R2, _TwoFactorBase.compute_Rp
    _dense_sums = _TwoFactorBase._dense_sums
    _up, _down = staticmethod(_TwoFactorBase._up), staticmethod(_TwoFactorBase._down)
    _set_scalars = _TwoFactorBase._set_scalars
    _init_trace_lists = _TwoFactorBase._init_trace_lists
    _run_loop = _TwoFactorBase._run_loop
    check_empty_rows_columns = _TwoFactorBase.check_empty_rows_columns

    def __init__(self, R, M, K, L, priors, device=None, seed=None):
        self._sparse = scipy.sparse.issparse(R)
        if self._sparse:
            # sparse input (as in the two-factor models): the stored entries of R are its known entries, explicit zeros
            # included; M (or None: all of them) selects the training entries; self.R / self.M are canonical CSR matrices
            self.R, self.M, self._train = validate_sparse(R, M)
            self.K = K
            self.L = L
            (self.I, self.J) = self.R.shape
            self.size_Omega = float(self.M.nnz)
        else:
            self.R = np.array(R, dtype=float)
            self.M = np.array(M, dtype=float)
            self.K = K
            self.L = L

            assert len(self.R.shape) == 2, "Input matrix R is not a two-dimensional array, " \
                "but instead %s-dimensional." % len(self.R.shape)
            assert self.R.shape == self.M.shape, "Input matrix R is not of the same size as " \
                "the indicator matrix M: %s and %s respectively." % (self.R.shape, self.M.shape)

            (self.I, self.J) = self.R.shape
            self.size_Omega = self.M.sum()
            self.check_empty_rows_columns()

        self.alpha, self.beta, self.lambdaF, self.lambdaS, self.lambdaG = \
            float(priors['alpha']), float(priors['beta']), np.array(priors['lambdaF']), np.array(priors['lambdaS']), np.array(priors['lambdaG'])
        if self.lambdaF.shape == ():
            self.lambdaF = self.lambdaF * np.ones((self.I, self.K))
        if self.lambdaS.shape == ():
            self.lambdaS = self.lambdaS * np.ones((self.K, self.L))
        if self.lambdaG.shape == ():
            self.lambdaG = self.lambdaG * np.ones((self.J, self.L))

        assert self.lambdaF.shape == (self.I, self.K), "Prior matrix lambdaF has the wrong shape: %s instead of (%s, %s)." % (self.lambdaF.shape, self.I, self.K)
        assert self.lambdaS.shape == (self.K, self.L), "Prior matrix lambdaS has the wrong shape: %s instead of (%s, %s)." % (self.lambdaS.shape, self.K, self.L)
        assert self.lambdaG.shape == (self.J, self.L), "Prior matrix lambdaG has the wrong shape: %s instead of (%s, %s)." % (self.lambdaG.shape, self.J, self.L)
        self._device_arg, self._seed, self._eng = device, seed, None
        self.verbose = False

    @classmethod
    def from_dataset(cls, dataset, K, L, priors, seed=None):
        """Build a model on an engine.Dataset / engine.SparseDataset that already lives on the GPU (matrices too large for,
        or never present in, host memory).  R and M stay None on the host.  init_FG='kmeans' works on a SparseDataset (it
        clusters the dataset's host CSR of the training entries), not on a dense Dataset."""
        self = cls.__new__(cls)
        self.R = self.M = None
        self._sparse = isinstance(dataset, SparseDataset)
        self.K, self.L = K, L
        (self.I, self.J) = (dataset.I, dataset.J)
        self.size_Omega = float(dataset.n_obs)
        self.alpha, self.beta = float(priors['alpha']), float(priors['beta'])
        for name, shape in (('lambdaF', (self.I, K)), ('lambdaS', (K, L)), ('lambdaG', (self.J, L))):
            lam = np.array(priors[name], dtype=float)
            setattr(self, name, lam * np.ones(shape) if lam.shape == () else lam)
        self._device_arg, self._seed, self.verbose = dataset.device, seed, False
        self._eng = tri_engine_for(dataset, K, L, cls._mode, self.alpha, self.beta,
                                   seed=seed if seed is not None else _lib.derive_seed())
        return self

    def _engine(self):
        if self._eng is None:
            dev = require_cuda(self._device_arg)
            if getattr(self, '_sparse', False):
                ds = SparseDataset(self.R, self._train, dev)
            else:
                ds = Dataset.from_host(self.R, self.M, dev)
            seed = self._seed if self._seed is not None else _lib.derive_seed()
            self._eng = tri_engine_for(ds, self.K, self.L, self._mode, self.alpha, self.beta, seed=seed)
        return self._eng

    def triple_dot(self, M1, M2, M3):
        dev = require_cuda(self._device_arg)
        a, b, c = (torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(dev) for x in (M1, M2, M3))
        bc = torch.empty((b.shape[0], c.shape[1]), dtype=torch.float64, device=dev)
        _lib.call("bnmtf_small_matmul_f64", _ptr(b), _ptr(c), b.shape[0], b.shape[1], c.shape[1], 0, _ptr(bc), _stream())
        out = torch.empty((a.shape[0], c.shape[1]), dtype=torch.float64, device=dev)
        _lib.call("bnmtf_small_matmul_f64", _ptr(a), _ptr(bc), a.shape[0], a.shape[1], c.shape[1], 0, _ptr(out), _stream())
        return out.cpu().numpy()

    def _n_params(self):
        return self.I * self.K + self.K * self.L + self.J * self.L

    _quality_from_ll = _TwoFactorBase._quality_from_ll

    def _sums_for(self, M_pred, F, S, G):
        eng = self._engine()
        self._up(eng.F.fac, F), self._up(eng.S["fac"], S), self._up(eng.G.fac, G)
        eng.metrics(None if M_pred is None else eng.ds.pack_mask(M_pred))
        return eng.m8.cpu().numpy()

    def _kmeans_init(self, offset):
        from .kmeans import KMeans, SparseKMeans
        dev = require_cuda(self._device_arg)            # the assignment step runs on the device (csrc/kmeans.cu)
        if getattr(self, '_sparse', False):
            # the observed entries only: the clusterings of KMeans on (R.toarray(), M.toarray()) and on their transposes
            if self.R is None:                          # from_dataset(SparseDataset)
                Xt, Xall = self._eng.ds.host_train, self._eng.ds.host_R
            else:
                Xt, Xall = training_csr(self.R, self._train), self.R
            kmeans_F = SparseKMeans(Xt, self.K, X_all=Xall, device=dev)
            kmeans_F.initialise()
            kmeans_F.cluster()
            kmeans_G = SparseKMeans(Xt.T.tocsr(), self.L, X_all=Xall.T.tocsr(), device=dev)
            kmeans_G.initialise()
            kmeans_G.cluster()
            return kmeans_F.clustering_results + offset, kmeans_G.clustering_results + offset
        kmeans_F = KMeans(self.R, self.M, self.K, device=dev)
        kmeans_F.initialise()
        kmeans_F.cluster()
        kmeans_G = KMeans(self.R.T, self.M.T, self.L, device=dev)
        kmeans_G.initialise()
        kmeans_G.cluster()
        return kmeans_F.clustering_results + offset, kmeans_G.clustering_results + offset


class _PointEstimateNMTF(_ThreeFactorBase):
    """Shared by the Gibbs sampler and ICM: state F, S, G, tau; conditionals tauF/muF, tauS/muS, tauG/muG."""

    def train(self, init_S, init_FG, iterations):
        self.initialise(init_S=init_S, init_FG=init_FG)   # the reference's train() passes a keyword its initialise lacks
        return self.run(iterations)

    def _initial_FSG(self, init_S, init_FG):
        assert init_S in ['random', 'exp'], "Unknown initialisation option for S: %s. Should be 'random' or 'exp'." % init_S
        assert init_FG in ['random', 'exp', 'kmeans'], "Unknown initialisation option for S: %s. Should be 'random', 'exp', or 'kmeans." % init_FG
        self.S = 1. / self.lambdaS
        if init_S == 'random':
            self.S = np.random.exponential(scale=1.0 / self.lambdaS)
        self.F, self.G = 1. / self.lambdaF, 1. / self.lambdaG
        if init_FG == 'random':
            self.F = np.random.exponential(scale=1.0 / self.lambdaF)
            self.G = np.random.exponential(scale=1.0 / self.lambdaG)
        elif init_FG == 'kmeans':
            self.F, self.G = self._kmeans_init(0.2)

    def _push(self):
        eng = self._engine()
        self._up(eng.F.fac, self.F), self._up(eng.S["fac"], self.S), self._up(eng.G.fac, self.G)
        self._up(eng.F.lam, self.lambdaF), self._up(eng.S["lam"], self.lambdaS), self._up(eng.G.lam, self.lambdaG)
        self._set_scalars(eng, {S_TAU: float(getattr(self, 'tau', 1.0))})
        return eng

    def alpha_s(self):
        return self.alpha + self.size_Omega / 2.0

    def beta_s(self):
        return self.beta + 0.5 * float(self._sums_for(None, self.F, self.S, self.G)[0])

    # conditional parameters of the current state (white-box API)
    def _outer_params(self, which, idx):
        eng = self._push()
        if which == 'F':
            eng.stats_rows()
            eng.phase_F(order=[idx], apply=False, want_sterm=True, use_iter=False)
            return self._down(eng.F.tauf)[:, idx], self._down(eng.sterm)[:, idx]
        eng.stats_cols()
        eng.phase_G(order=[idx], apply=False, want_sterm=True, use_iter=False)
        return self._down(eng.G.tauf)[:, idx], self._down(eng.sterm)[:, idx]

    def tauF(self, k):
        return self._outer_params('F', k)[0]

    def muF(self, tauFk, k):
        s = self._outer_params('F', k)[1]
        with np.errstate(all='ignore'):
            return 1. / np.asarray(tauFk) * (-self.lambdaF[:, k] + self.tau * s)

    def tauG(self, l):
        return self._outer_params('G', l)[0]

    def muG(self, tauGl, l):
        s = self._outer_params('G', l)[1]
        with np.errstate(all='ignore'):
            return 1. / np.asarray(tauGl) * (-self.lambdaG[:, l] + self.tau * s)

    def _s_params(self, k, l):
        eng = self._push()
        eng.stats_rows()
        eng.phase_S(order=[k * self.L + l], apply=False, use_iter=False)
        tau_kl = float(self._down(eng.S["tauf"])[k, l])
        mu_kl = float(self._down(eng.S["mu"])[k, l])
        return tau_kl, mu_kl

    def tauS(self, k, l):
        return self._s_params(k, l)[0]

    def muS(self, tauSkl, k, l):
        tau_kl, mu_kl = self._s_params(k, l)
        s = (mu_kl * tau_kl + self.lambdaS[k, l]) / self.tau      # the masked-sum term the kernel used
        with np.errstate(all='ignore'):
            return 1. / tauSkl * (-self.lambdaS[k, l] + self.tau * s)

    def _pull_state(self, eng, tr, iterations):
        self.F, self.S, self.G = self._down(eng.F.fac), self._down(eng.S["fac"]), self._down(eng.G.fac)
        self.all_tau = tr[:, 0].copy()
        if iterations > 0:
            self.tau = float(tr[-1, 0])


class bnmtf_gibbs_optimised(_PointEstimateNMTF):
    """Gibbs sampler for BNMTF (reference code/models/bnmtf_gibbs_optimised.py)."""
    _mode = 'gibbs'

    def initialise(self, init_S='random', init_FG='random'):
        self._initial_FSG(init_S, init_FG)
        self.tau = self.alpha_s() / self.beta_s()

    def run(self, iterations):
        eng = self._push()
        dev = eng.ds.device
        z = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
        all_F, all_S, all_G = z(iterations, self.I, self.K), z(iterations, self.K, self.L), z(iterations, self.J, self.L)
        self._init_trace_lists()

        def keep(it):
            all_F[it].copy_(eng.F.fac), all_S[it].copy_(eng.S["fac"]), all_G[it].copy_(eng.G.fac)
        tr = self._run_loop(eng, iterations, per_iteration=keep, samples=(all_F, all_S, all_G))
        self.all_F, self.all_S, self.all_G = self._down(all_F), self._down(all_S), self._down(all_G)
        self._pull_state(eng, tr, iterations)
        return (self.all_F, self.all_S, self.all_G, self.all_tau)

    def approx_expectation(self, burn_in, thinning):
        indices = range(burn_in, len(self.all_F), thinning)
        n = float(len(indices))
        exp_F = np.array([self.all_F[i] for i in indices]).sum(axis=0) / n
        exp_S = np.array([self.all_S[i] for i in indices]).sum(axis=0) / n
        exp_G = np.array([self.all_G[i] for i in indices]).sum(axis=0) / n
        exp_tau = sum([self.all_tau[i] for i in indices]) / n
        return (exp_F, exp_S, exp_G, exp_tau)

    def predict(self, M_pred, burn_in, thinning):
        (exp_F, exp_S, exp_G, _) = self.approx_expectation(burn_in, thinning)
        return _metrics_from_sums(self._sums_for(M_pred, exp_F, exp_S, exp_G))

    def predict_while_running(self):
        return _metrics_from_sums(self._sums_for(None, self.F, self.S, self.G))

    def quality(self, metric, burn_in, thinning):
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        (expF, expS, expG, exptau) = self.approx_expectation(burn_in, thinning)
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, expF, expS, expG))['MSE']
        elif metric == 'ELBO':
            return 0.
        return self._quality_from_ll(metric, self.log_likelihood(expF, expS, expG, exptau))

    def log_likelihood(self, expF, expS, expG, exptau):
        explogtau = math.log(exptau)
        return self.size_Omega / 2. * (explogtau - math.log(2 * math.pi)) \
            - exptau / 2. * float(self._sums_for(None, expF, expS, expG)[0])


class nmtf_icm(_PointEstimateNMTF):
    """Iterated conditional modes for NMTF (reference code/models/nmtf_icm.py)."""
    _mode = 'icm'

    def initialise(self, init_S='random', init_FG='random'):
        self._initial_FSG(init_S, init_FG)
        self.tau = (self.alpha_s() - 1.) / self.beta_s()

    def run(self, iterations, minimum_TN=0.):
        eng = self._push()
        self._init_trace_lists()
        tr = self._run_loop(eng, iterations, minimum_TN=minimum_TN)
        self._pull_state(eng, tr, iterations)
        return

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums_for(M_pred, self.F, self.S, self.G))

    def quality(self, metric):
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, self.F, self.S, self.G))['MSE']
        elif metric == 'ELBO':
            return 0.
        return self._quality_from_ll(metric, self.log_likelihood())

    def log_likelihood(self):
        return self.size_Omega / 2. * (math.log(self.tau) - math.log(2 * math.pi)) \
            - self.tau / 2. * float(self._sums_for(None, self.F, self.S, self.G)[0])


# =====================================================================================================
class bnmtf_vb_optimised(_ThreeFactorBase):
    """Variational Bayes for BNMTF (reference code/models/bnmtf_vb_optimised.py)."""
    _mode = 'vb'

    def train(self, init_S, init_FG, iterations):
        self.initialise(init_S, init_FG)
        return self.run(iterations)

    def initialise(self, init_S='random', init_FG='random', tauFSG={}):
        self.tauF = tauFSG['tauF'] if 'tauF' in tauFSG else np.ones((self.I, self.K))
        self.tauS = tauFSG['tauS'] if 'tauS' in tauFSG else np.ones((self.K, self.L))
        self.tauG = tauFSG['tauG'] if 'tauG' in tauFSG else np.ones((self.J, self.L))
        assert init_S in ['exp', 'random'], "Unrecognised init option for S: %s." % init_S
        self.muS = 1. / self.lambdaS
        if init_S == 'random':
            self.muS = np.random.exponential(scale=1.0 / self.lambdaS)
        assert init_FG in ['exp', 'random', 'kmeans'], "Unrecognised init option for F,G: %s." % init_FG
        self.muF, self.muG = 1. / self.lambdaF, 1. / self.lambdaG
        if init_FG == 'random':
            self.muF = np.random.exponential(scale=1.0 / self.lambdaF)
            self.muG = np.random.exponential(scale=1.0 / self.lambdaG)
        elif init_FG == 'kmeans':
            self.muF, self.muG = self._kmeans_init(0.0)
        # (the reference's update_exp_F / update_exp_S / update_exp_G loops, :141-146, as one device call per factor: the
        # moments are element-wise)
        from .distributions import TN_matrix_moments
        self.expF, self.varF = TN_matrix_moments(self.muF, self.tauF)
        self.expS, self.varS = TN_matrix_moments(self.muS, self.tauS)
        self.expG, self.varG = TN_matrix_moments(self.muG, self.tauG)
        self.update_tau()
        self.update_exp_tau()

    def _push(self):
        eng = self._engine()
        # (attributes the caller has not set yet are not uploaded -- see bnmf.bnmf_vb_optimised._push)
        for f, s in ((eng.F, 'F'), (eng.G, 'G')):
            for attr, t in (('exp', f.fac), ('var', f.var), ('mu', f.mu), ('tau', f.tauf)):
                value = getattr(self, attr + s, None)
                if value is not None:
                    self._up(t, value)
            self._up(f.lam, getattr(self, 'lambda' + s))
        S = eng.S
        for attr, key in (('exp', 'fac'), ('var', 'var'), ('mu', 'mu'), ('tau', 'tauf')):
            value = getattr(self, attr + 'S', None)
            if value is not None:
                self._up(S[key], value)
        self._up(S["lam"], self.lambdaS)
        self._set_scalars(eng, {S_TAU: float(getattr(self, 'exptau', 1.0)), S_LOGTAU: float(getattr(self, 'explogtau', 0.0)),
                                S_BETA_S: float(getattr(self, 'beta_s', 1.0))})
        return eng

    def _pull(self, eng):
        for f, s in ((eng.F, 'F'), (eng.G, 'G')):
            for attr, t in (('exp', f.fac), ('var', f.var), ('mu', f.mu), ('tau', f.tauf)):
                setattr(self, attr + s, self._down(t))
        for attr, key in (('exp', 'fac'), ('var', 'var'), ('mu', 'mu'), ('tau', 'tauf')):
            setattr(self, attr + 'S', self._down(eng.S[key]))

    def run(self, iterations):
        eng = self._push()
        self._init_trace_lists()
        K, L = self.K, self.L
        eng.alloc_trace(iterations)

        def shuffles():
            # the reference's three python-`random` shuffles, in its call order (bnmtf_vb_optimised.py:171-190)
            indices_kl = list(itertools.product(range(0, K), range(0, L)))
            random.shuffle(indices_kl)
            indices_k = list(range(0, K))
            random.shuffle(indices_k)
            indices_l = list(range(0, L))
            random.shuffle(indices_l)
            return [k * L + l for k, l in indices_kl], indices_k, indices_l
        # the orders of every sweep are drawn up front, in the reference's call order (three shuffles per iteration)
        todo = [shuffles() for _ in range(iterations)]
        launched = False
        if iterations > 0 and eng.small_cluster():
            # small matrix: the whole run is one kernel (csrc/small.cu::k_small_tri)
            od = torch.from_numpy(np.array([oS + oF + oG for oS, oF, oG in todo], dtype=np.int32)).to(eng.ds.device)
            times = torch.zeros(iterations + 1, dtype=torch.int64, device=eng.ds.device)
            try:
                eng.sweep_many(iterations, 0.0, None, times, None, od)
                launched = True
            except _lib.BnmtfError as exc:
                import warnings
                warnings.warn("bnmtf_b200: single-kernel sweep not launched (%s); using the per-phase kernels" % exc)
                eng._small_c = 0
            if launched:
                torch.cuda.synchronize()
                t = times.cpu().numpy()
                self.all_times = [float(x - t[0]) / 1e9 for x in t[1:]]
        if not launched:
            start = torch.cuda.Event(enable_timing=True)
            marks = []
            start.record()
            for oS, oF, oG in todo:
                eng.sweep(order={"S": oS, "F": oF, "G": oG})
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append(ev)
            torch.cuda.synchronize()
            self.all_times = [start.elapsed_time(ev) / 1e3 for ev in marks]
        tr = eng.trace.cpu().numpy()[:iterations]
        for i, metric in enumerate(METRICS):
            self.all_performances[metric] = [float(v) for v in tr[:, 1 + i]]
        self.all_exp_tau = [float(v) for v in tr[:, 0]]
        self.all_elbo = [float(v) for v in tr[:, 4]]
        self._pull(eng)
        if iterations > 0:
            sc = eng.scalars.cpu().numpy()
            self.exptau, self.explogtau = float(sc[S_TAU]), float(sc[S_LOGTAU])
            self.alpha_s, self.beta_s = self.alpha + self.size_Omega / 2.0, float(sc[S_BETA_S])
        return

    # ---- white-box pieces -----------------------------------------------------------------------------------
    def _refreshed_scalars(self, update_tau):
        eng = self._push()
        eng.refresh_scalars(update_tau=update_tau)
        return eng.scalars.cpu().numpy()

    def elbo(self):
        return float(self._refreshed_scalars(False)[S_ELBO]) + _elbo_alpha_s_correction(self)

    def exp_square_diff(self):
        return float(self._refreshed_scalars(False)[S_ESD])

    def update_tau(self):
        self.alpha_s = self.alpha + self.size_Omega / 2.0
        self.beta_s = self.beta + 0.5 * self.exp_square_diff()

    def update_exp_tau(self):
        from scipy.special import psi
        self.exptau = float(self.alpha_s) / float(self.beta_s)
        self.explogtau = float(psi(float(self.alpha_s))) - math.log(float(self.beta_s))

    def update_F(self, k):
        eng = self._push()
        eng.stats_rows()
        eng.phase_F(order=[k], apply=False, use_iter=False)
        self.tauF[:, k], self.muF[:, k] = self._down(eng.F.tauf)[:, k], self._down(eng.F.mu)[:, k]

    def update_G(self, l):
        eng = self._push()
        eng.stats_cols()
        eng.phase_G(order=[l], apply=False, use_iter=False)
        self.tauG[:, l], self.muG[:, l] = self._down(eng.G.tauf)[:, l], self._down(eng.G.mu)[:, l]

    def update_S(self, k, l):
        eng = self._push()
        eng.stats_rows()
        eng.phase_S(order=[k * self.L + l], apply=False, use_iter=False)
        self.tauS[k, l], self.muS[k, l] = self._down(eng.S["tauf"])[k, l], self._down(eng.S["mu"])[k, l]

    def update_exp_F(self, k):
        from .distributions import TN_vector_expectation, TN_vector_variance
        self.expF[:, k] = TN_vector_expectation(self.muF[:, k], self.tauF[:, k])
        self.varF[:, k] = TN_vector_variance(self.muF[:, k], self.tauF[:, k])

    def update_exp_S(self, k, l):
        from .distributions import TN_expectation, TN_variance
        self.expS[k, l] = TN_expectation(self.muS[k, l], self.tauS[k, l])
        self.varS[k, l] = TN_variance(self.muS[k, l], self.tauS[k, l])

    def update_exp_G(self, l):
        from .distributions import TN_vector_expectation, TN_vector_variance
        self.expG[:, l] = TN_vector_expectation(self.muG[:, l], self.tauG[:, l])
        self.varG[:, l] = TN_vector_variance(self.muG[:, l], self.tauG[:, l])

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums_for(M_pred, self.expF, self.expS, self.expG))

    def quality(self, metric):
        metric = 'ELBO' if metric == 'elbo' else metric
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, self.expF, self.expS, self.expG))['MSE']
        elif metric == 'ELBO':
            return self.elbo()
        return self._quality_from_ll(metric, self.log_likelihood())

    def log_likelihood(self):
        return self.size_Omega / 2. * (self.explogtau - math.log(2 * math.pi)) \
            - self.exptau / 2. * float(self._sums_for(None, self.expF, self.expS, self.expG)[0])


BNMTF_Gibbs = bnmtf_gibbs_optimised
BNMTF_VB = bnmtf_vb_optimised
