"""Drop-in classes for the reference's non-probabilistic models:

    NMF   (code/models/nmf_np.py:32)   -- Lee & Seung multiplicative updates (I-divergence) with a mask
    NMTF  (code/models/nmtf_np.py:39)  -- Yoo & Choi multiplicative tri-factorisation with a mask

Same constructor / initialise / run / train / update_* / predict / compute_I_div surface as the reference.  On dense
input the prediction matrix lives in a device scratch buffer (csrc/np.cu); on sparse input (a scipy.sparse R) only the
observed entries exist on the device (csrc/sparse_np.cu).  Every update is a CUDA kernel.
"""
import itertools
import time

import numpy as np
import scipy.sparse
import torch

from . import _lib
from .bnmf import _metrics_from_sums
from .data import validate_sparse
from .engine import CSR_METRIC_CTAS, Dataset, SparseDataset, _ptr, _stream, require_cuda

# Row classes of the sparse row update (bnmtf_csr_np_row_update_f64): a warp holds up to 8 entries per lane in registers,
# a CTA of 256 threads up to 8 per thread; longer rows go to clusters of 2..16 CTAs, each with about NP_CTA_MAX entries
NP_WARP_MAX = 256
NP_CTA_MAX = 2048
NP_CLUSTER_MAX = 16
NP_S_CTAS = 592         # CTAs (partial results) of one S-phase launch: 4 per SM


def _mm(A, B, transB):
    """A B (or A B^T) of factor-sized device matrices with bnmtf_small_matmul_f64."""
    n, p = A.shape
    q = B.shape[0] if transB else B.shape[1]
    C = torch.empty((n, q), dtype=torch.float64, device=A.device)
    _lib.call("bnmtf_small_matmul_f64", _ptr(A), _ptr(B), n, p, q, 1 if transB else 0, _ptr(C), _stream())
    return C


def np_row_plan(indptr):
    """Static work plan of bnmtf_csr_np_row_update_f64 for the row pointers `indptr` (include/bnmtf_b200.h): rows of at
    most NP_WARP_MAX entries become warp items, rows of at most NP_CTA_MAX CTA items, longer rows nc cluster items (nc the
    power of two >= ceil(n / NP_CTA_MAX), at most NP_CLUSTER_MAX), each a contiguous range of ceil(n / nc) entries in rank
    order.  -> dict of numpy arrays item_row (int32), item_beg, item_end (int64) in class order, and `counts`: the item
    count of each class (warp, CTA, clusters of 2, 4, 8, 16)."""
    indptr = np.asarray(indptr, dtype=np.int64)
    lens = np.diff(indptr)
    rows = np.arange(lens.shape[0], dtype=np.int64)
    need = -(-lens // NP_CTA_MAX)
    nc = np.minimum(NP_CLUSTER_MAX, 1 << np.ceil(np.log2(np.maximum(need, 1))).astype(np.int64))
    classes = [rows[lens <= NP_WARP_MAX], rows[(lens > NP_WARP_MAX) & (lens <= NP_CTA_MAX)]]
    heavy = lens > NP_CTA_MAX
    parts_row, parts_beg, parts_end, counts = [], [], [], [len(c) for c in classes]
    for r in classes:
        parts_row.append(r), parts_beg.append(indptr[r]), parts_end.append(indptr[r + 1])
    for c in (2, 4, 8, 16):
        r = rows[heavy & (nc == c)]
        q = np.tile(np.arange(c, dtype=np.int64), r.shape[0])
        rr = np.repeat(r, c)
        share = -(-lens[rr] // c)
        parts_row.append(rr)
        parts_beg.append(np.minimum(indptr[rr] + q * share, indptr[rr + 1]))
        parts_end.append(np.minimum(indptr[rr] + (q + 1) * share, indptr[rr + 1]))
        counts.append(int(rr.shape[0]))
    return {"item_row": np.concatenate(parts_row).astype(np.int32), "item_beg": np.concatenate(parts_beg),
            "item_end": np.concatenate(parts_end), "counts": counts}


def _check_width(name, v):
    if not 1 <= int(v) <= 63:
        raise ValueError("%s=%s out of range (1..63)" % (name, v))


class _NPEngine:
    """Device buffers shared by NMF and NMTF on dense input: the dataset in both orientations, the prediction P = A B^T in
    both orientations (rebuilt at the start of each phase), reduction scratch."""

    def __init__(self, ds):
        self.ds = ds
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=ds.device)
        self.P = f64(ds.I, ds.ldJ)
        self.PT = f64(ds.J, ds.ldI)
        self.nparts = 128
        self.part = f64(self.nparts * 8 + 8)
        self.out8 = f64(8)

    def dev(self, x):
        return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(self.ds.device)

    def build_pred(self, A, B, transposed=False):
        ds = self.ds
        if transposed:   # PT = B A^T : rows J
            _lib.call("bnmtf_np_build_pred_f64", _ptr(B), _ptr(A), ds.J, ds.I, ds.ldI, A.shape[1], _ptr(self.PT), _stream())
        else:
            _lib.call("bnmtf_np_build_pred_f64", _ptr(A), _ptr(B), ds.I, ds.J, ds.ldJ, A.shape[1], _ptr(self.P), _stream())

    def row_update(self, A, B, transposed=False):
        """All columns of A (rows of R, or of R^T when transposed) against B; P / PT must be current."""
        ds = self.ds
        if transposed:
            _lib.call("bnmtf_np_row_update_f64", _ptr(ds.RT), _ptr(ds.bitsT), _ptr(self.PT), ds.J, ds.I, ds.ldI,
                      _ptr(A), _ptr(B), A.shape[1], _stream())
        else:
            _lib.call("bnmtf_np_row_update_f64", _ptr(ds.R), _ptr(ds.bits), _ptr(self.P), ds.I, ds.J, ds.ldJ,
                      _ptr(A), _ptr(B), A.shape[1], _stream())

    # ---- the model classes' device calls -------------------------------------------------------------------
    def phase(self, A, B, transposed=False, k0=0, k1=None):
        """Columns k0..k1-1 (default: all) of A, in order, against B: the rows of R (R^T when transposed)."""
        if transposed:
            self.build_pred(B, A, transposed=True)
        else:
            self.build_pred(A, B)
        if k1 is None:
            self.row_update(A, B, transposed)
        else:
            for k in range(k0, k1):
                a, b = A[:, k:k + 1].contiguous(), B[:, k:k + 1].contiguous()
                self.row_update(a, b, transposed)
                A[:, k] = a[:, 0]

    def s_phase(self, F, S, G, pairs):
        """NMTF's S updates over the (k, l) pairs in order."""
        ds = self.ds
        K, L = F.shape[1], G.shape[1]
        self.build_pred(_mm(F, S, False), G)
        for k, l in pairs:
            _lib.call("bnmtf_np_s_update_f64", _ptr(ds.R), _ptr(ds.bits), _ptr(self.P), ds.I, ds.J, ds.ldJ, _ptr(F), K, k,
                      _ptr(G), L, l, _ptr(S), _ptr(self.part), self.nparts, _stream())

    def sums(self, A, B, M_pred=None):
        """The eight sums of the prediction A B^T over the training entries (M_pred None) or M_pred's -> numpy."""
        ds = self.ds
        self.build_pred(A, B)
        bits = ds.bits if M_pred is None else ds.pack_mask(M_pred)
        _lib.call("bnmtf_np_metrics_f64", _ptr(ds.R), _ptr(bits), _ptr(self.P), ds.I, ds.J,
                  ds.ldJ, _ptr(self.part), self.nparts, _ptr(self.out8), _stream())
        return self.out8.cpu().numpy()

    def sums_into(self, A, B, trace, row):
        """The eight masked sums of the prediction A B^T -> trace[row] on the device (no host round trip)."""
        ds = self.ds
        self.build_pred(A, B)
        _lib.call("bnmtf_np_metrics_f64", _ptr(ds.R), _ptr(ds.bits), _ptr(self.P), ds.I, ds.J, ds.ldJ, _ptr(self.part),
                  self.nparts, _ptr(trace, row), _stream())

    def run_loop(self, iterations, body):
        """iterations x body() with the per-iteration sums of the prediction body() returns (A, B: P = A B^T) kept in a
        device trace and CUDA events for all_times; the launch sequence of an iteration has fixed arguments except the
        trace row, which advances through a device-side pointer table -- so it is captured once and replayed as a CUDA
        graph (these problems are launch-latency-bound).  Returns (trace as numpy, cumulative seconds per iteration)."""
        import os
        from .engine import capture_graph, thread_flags
        dev = self.ds.device
        trace = torch.zeros((max(1, iterations), 8), dtype=torch.float64, device=dev)
        start = torch.cuda.Event(enable_timing=True)
        marks = []
        use_graph = int(os.environ.get("BNMTF_GRAPH", "1")) >= 1 and not getattr(thread_flags, "no_graph", False) and iterations >= 8
        graph = None
        start.record()
        for it in range(iterations):
            if use_graph and it >= 1:
                # iterations 1.. write their sums to the scratch row out8; a tiny copy moves them to trace[it] afterwards
                if graph is None:
                    count0 = _lib.launch_count[0]

                    def captured():
                        self.sums_into(*body(), self.out8.view(1, 8), 0)
                    graph = capture_graph(captured)
                    self._graph_kernels = _lib.launch_count[0] - count0
                    _lib.launch_count[0] = count0
                graph.replay()
                _lib.launch_count[0] += self._graph_kernels
                trace[it].copy_(self.out8)
            else:
                self.sums_into(*body(), trace, it)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
        torch.cuda.synchronize()
        return trace.cpu().numpy()[:iterations], [start.elapsed_time(ev) / 1e3 for ev in marks]


class _SparseNPEngine(_NPEngine):
    """The same device calls on a SparseDataset (csrc/sparse_np.cu): the one place that knows the sparse format.  The
    prediction exists only per observed entry -- in registers, or in the per-entry scratch `pw` for the heavy rows of
    the row update and for the S phase.  run_loop (CUDA-graph replay) is _NPEngine's."""

    def __init__(self, ds):
        self.ds = ds
        dev = ds.device
        self.plan = {}
        for side in (0, 1):
            p = np_row_plan(ds.csr[side].rowptr.cpu().numpy())
            t = lambda a: torch.from_numpy(a).to(dev)
            self.plan[side] = (t(p["item_beg"]), t(p["item_end"]), t(p["item_row"]), p["counts"])
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
        self.pw = f64(max(1, ds.csr[0].nnz))
        self.nparts = NP_S_CTAS
        self.part = f64(max(CSR_METRIC_CTAS * 8, 4 * NP_S_CTAS + 2))
        self.out8 = f64(8)
        self._pairs = {}

    def phase(self, A, B, transposed=False, k0=0, k1=None):
        side = 1 if transposed else 0
        c = self.ds.csr[side]
        beg, end, row, counts = self.plan[side]
        k1 = A.shape[1] if k1 is None else k1
        _lib.call("bnmtf_csr_np_row_update_f64", _ptr(beg), _ptr(end), _ptr(row), *counts, _ptr(c.colidx), _ptr(c.val),
                  _ptr(A), _ptr(B), A.shape[1], k0, k1, _ptr(self.pw), _stream())
        _lib.launch_count[0] += sum(1 for n in counts if n)

    def s_phase(self, F, S, G, pairs):
        key = tuple(pairs)
        if key not in self._pairs:       # first use is outside graph capture (run_loop's iteration 0 runs eagerly)
            self._pairs[key] = torch.tensor(np.asarray(pairs, dtype=np.int32).reshape(-1), device=self.ds.device)
        c = self.ds.csr[0]
        _lib.call("bnmtf_csr_np_s_update_f64", _ptr(c.rowptr), _ptr(c.colidx), _ptr(c.val), _ptr(c.item_begin),
                  _ptr(c.item_row), c.n_items, c.chunk, _ptr(_mm(F, S, False)), _ptr(F), F.shape[1], _ptr(G), G.shape[1],
                  _ptr(self._pairs[key]), len(pairs), _ptr(S), _ptr(self.pw), _ptr(self.part), self.nparts, _stream())
        _lib.launch_count[0] += len(pairs)

    def _metrics(self, A, B, entries, out):
        nparts = max(1, min(CSR_METRIC_CTAS, -(-entries.rows // 8)))
        _lib.call("bnmtf_csr_np_metrics_f64", _ptr(entries.rowptr), _ptr(entries.colidx), _ptr(entries.val), entries.rows,
                  _ptr(A), _ptr(B), A.shape[1], _ptr(self.part), nparts, _ptr(out), _stream())

    def sums(self, A, B, M_pred=None):
        self._metrics(A, B, self.ds.csr[0] if M_pred is None else self.ds.pack_mask(M_pred), self.out8)
        return self.out8.cpu().numpy()

    def sums_into(self, A, B, trace, row):
        self._metrics(A, B, self.ds.csr[0], trace[row])


def _engine_for(ds):
    if ds.world != 1:
        raise ValueError("the NP models run on one GPU: the dataset must not be sharded")
    return _SparseNPEngine(ds) if isinstance(ds, SparseDataset) else _NPEngine(ds)


class _NPBase(object):
    def _common_init(self, R, M, device):
        self._sparse = scipy.sparse.issparse(R)
        self.metrics = ['MSE', 'R^2', 'Rp']
        self._device_arg, self._eng = device, None
        self.verbose = False
        if self._sparse:
            # the stored entries of R are its known entries, explicit zeros included; M (or None: all of them) selects
            # the training entries; self.R / self.M are canonical CSR matrices.  R_excl_unknown (I x J) is not built.
            self.R, self.M, self._train = validate_sparse(R, M)
            (self.I, self.J) = self.R.shape
            return
        if scipy.sparse.issparse(M):
            raise ValueError("with dense R, M must be a dense array, not %s" % type(M).__name__)
        self.R = np.array(R, dtype=float)
        self.M = np.array(M, dtype=float)
        self.metrics = ['MSE', 'R^2', 'Rp']
        assert len(self.R.shape) == 2, "Input matrix R is not a two-dimensional array, " \
            "but instead %s-dimensional." % len(self.R.shape)
        assert self.R.shape == self.M.shape, "Input matrix R is not of the same size as " \
            "the indicator matrix M: %s and %s respectively." % (self.R.shape, self.M.shape)
        (self.I, self.J) = self.R.shape
        self.check_empty_rows_columns()
        # For computing the I-div it is better if unknown values are 1's, not 0's (reference nmf_np.py:48-51)
        self.R_excl_unknown = np.where(self.M != 0, self.R, 1.)

    def _from_dataset(self, dataset):
        self.R = self.M = None
        self._sparse = isinstance(dataset, SparseDataset)
        (self.I, self.J) = (dataset.I, dataset.J)
        self.metrics = ['MSE', 'R^2', 'Rp']
        self._device_arg, self.verbose = dataset.device, False
        self._eng = _engine_for(dataset)

    def check_empty_rows_columns(self):
        sums_columns = self.M.sum(axis=0)
        sums_rows = self.M.sum(axis=1)
        for i, c in enumerate(sums_rows):
            assert c != 0, "Fully unobserved row in R, row %s." % i
        for j, c in enumerate(sums_columns):
            assert c != 0, "Fully unobserved column in R, column %s." % j

    def _engine(self):
        if self._eng is None:
            dev = require_cuda(self._device_arg)
            if self._sparse:
                self._eng = _SparseNPEngine(SparseDataset(self.R, self._train, dev))
            else:
                self._eng = _NPEngine(Dataset.from_host(self.R, self.M, dev))
        return self._eng

    def _dense_sums(self, M, R, R_pred):
        dev = require_cuda(self._device_arg)
        t = [torch.from_numpy(np.ascontiguousarray(np.broadcast_to(x, np.shape(R)), dtype=np.float64)).to(dev) for x in (R, R_pred, M)]
        part = torch.zeros(64 * 8, dtype=torch.float64, device=dev)
        out = torch.zeros(8, dtype=torch.float64, device=dev)
        _lib.call("bnmtf_dense_metrics_f64", _ptr(t[0]), _ptr(t[1]), _ptr(t[2]), t[0].numel(), _ptr(part), 64, _ptr(out), _stream())
        return out.cpu().numpy()

    def compute_MSE(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['MSE']

    def compute_R2(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['R^2']

    def compute_Rp(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['Rp']

    def _start_run(self):
        self.all_times = []
        self.all_performances = {}
        for metric in self.metrics:
            self.all_performances[metric] = []
        self.all_i_div = []

    def _record(self, sums, iteration, seconds):
        perf = _metrics_from_sums(sums)
        for metric in self.metrics:
            self.all_performances[metric].append(perf[metric])
        self.all_i_div.append(float(sums[7]))
        if self.verbose:
            print("Iteration %s. I-divergence: %s. MSE: %s. R^2: %s. Rp: %s." % (iteration, sums[7], perf['MSE'], perf['R^2'], perf['Rp']))
        self.all_times.append(seconds)


class NMF(_NPBase):
    def __init__(self, R, M, K, device=None):
        self.K = K
        self._common_init(R, M, device)
        if self._sparse:
            _check_width("K", K)

    @classmethod
    def from_dataset(cls, dataset, K):
        """NMF on an engine.SparseDataset (data.upload_sparse) or a single-GPU engine.Dataset that already lives on the
        GPU, so that several models share one resident copy of the matrix.  R and M stay None on the host."""
        _check_width("K", K)
        self = cls.__new__(cls)
        self.K = K
        self._from_dataset(dataset)
        return self

    def initialise(self, init_UV='random', expo_prior=1.):
        assert init_UV in ['ones', 'random', 'exponential'], "Unrecognised init option for U,V: %s." % init_UV
        if init_UV == 'ones':
            self.U = np.ones((self.I, self.K))
            self.V = np.ones((self.J, self.K))
        elif init_UV == 'random':
            self.U = np.random.rand(self.I, self.K)
            self.V = np.random.rand(self.J, self.K)
        elif init_UV == 'exponential':
            self.U = np.random.exponential(scale=1.0 / expo_prior, size=(self.I, self.K))
            self.V = np.random.exponential(scale=1.0 / expo_prior, size=(self.J, self.K))

    def run(self, iterations):
        assert hasattr(self, 'U') and hasattr(self, 'V'), "U and V have not been initialised - please run NMF.initialise() first."
        eng = self._engine()
        U, V = eng.dev(self.U), eng.dev(self.V)
        self._start_run()

        def body():
            eng.phase(U, V)
            eng.phase(V, U, transposed=True)
            return U, V
        trace, secs = eng.run_loop(iterations, body)
        for it in range(iterations):
            self._record(trace[it], it + 1, secs[it])
        self.U, self.V = U.cpu().numpy(), V.cpu().numpy()

    def train(self, iterations, init_UV='random', expo_prior=1.):
        self.initialise(init_UV=init_UV, expo_prior=expo_prior)
        self.run(iterations=iterations)

    def update_U(self, k):
        self._column(k, 'U')

    def update_V(self, k):
        self._column(k, 'V')

    def _column(self, k, side):
        """White-box single-column update of U[:, k] or V[:, k] with the prediction of the current U, V."""
        eng = self._engine()
        U, V = eng.dev(self.U), eng.dev(self.V)
        if side == 'U':
            eng.phase(U, V, k0=k, k1=k + 1)
            self.U[:, k] = U[:, k].cpu().numpy()
        else:
            eng.phase(V, U, transposed=True, k0=k, k1=k + 1)
            self.V[:, k] = V[:, k].cpu().numpy()

    def _sums(self, M_pred=None):
        eng = self._engine()
        return eng.sums(eng.dev(self.U), eng.dev(self.V), M_pred)

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums(M_pred))

    def compute_I_div(self):
        return float(self._sums()[7])

    def give_update(self, iteration):
        sums = self._sums()
        if not hasattr(self, 'all_performances'):
            self._start_run()
        self._record(sums, iteration, time.time())


class NMTF(_NPBase):
    def __init__(self, R, M, K, L, device=None):
        self.K = K
        self.L = L
        self._common_init(R, M, device)
        if self._sparse:
            _check_width("K", K), _check_width("L", L)

    @classmethod
    def from_dataset(cls, dataset, K, L):
        """NMTF on an engine.SparseDataset (data.upload_sparse) or a single-GPU engine.Dataset that already lives on the
        GPU, so that several models share one resident copy of the matrix.  R and M stay None on the host; init_FG='kmeans'
        needs a SparseDataset (it clusters the dataset's host CSR of the training entries)."""
        _check_width("K", K), _check_width("L", L)
        self = cls.__new__(cls)
        self.K, self.L = K, L
        self._from_dataset(dataset)
        return self

    def initialise(self, init_S='random', init_FG='random', expo_prior=1.):
        assert init_S in ['ones', 'random', 'exponential'], "Unrecognised init option for S: %s." % init_S
        assert init_FG in ['ones', 'random', 'exponential', 'kmeans'], "Unrecognised init option for F,G: %s." % init_FG
        if init_S == 'ones':
            self.S = np.ones((self.K, self.L))
        elif init_S == 'random':
            self.S = np.random.rand(self.K, self.L)
        elif init_S == 'exponential':
            self.S = np.random.exponential(scale=1.0 / expo_prior, size=(self.K, self.L))
        if init_FG == 'ones':
            self.F = np.ones((self.I, self.K))
            self.G = np.ones((self.J, self.L))
        elif init_FG == 'random':
            self.F = np.random.rand(self.I, self.K)
            self.G = np.random.rand(self.J, self.L)
        elif init_FG == 'exponential':
            self.F = np.random.exponential(scale=1.0 / expo_prior, size=(self.I, self.K))
            self.G = np.random.exponential(scale=1.0 / expo_prior, size=(self.J, self.L))
        elif init_FG == 'kmeans' and self._sparse:
            # the observed entries only (SparseKMeans), as the Bayesian tri-factor models do: the dense K-means results
            from .bnmtf import _ThreeFactorBase
            self.F, self.G = _ThreeFactorBase._kmeans_init(self, 0.2)
        elif init_FG == 'kmeans':
            from .kmeans import KMeans
            kmeans_F = KMeans(self.R, self.M, self.K)
            kmeans_F.initialise()
            kmeans_F.cluster()
            self.F = kmeans_F.clustering_results + 0.2
            kmeans_G = KMeans(self.R.T, self.M.T, self.L)
            kmeans_G.initialise()
            kmeans_G.cluster()
            self.G = kmeans_G.clustering_results + 0.2

    # ---- device pieces ---------------------------------------------------------------------------------------
    _mm = staticmethod(_mm)

    def _phase_F(self, eng, F, S, G, single=None):
        X = _mm(G, S, True)                   # J x K : (S G^T)^T
        eng.phase(F, X, k0=0 if single is None else single, k1=None if single is None else single + 1)

    def _phase_G(self, eng, F, S, G, single=None):
        X = _mm(F, S, False)                  # I x L : F S
        eng.phase(G, X, transposed=True, k0=0 if single is None else single, k1=None if single is None else single + 1)

    def _state(self):
        eng = self._engine()
        return eng, eng.dev(self.F), eng.dev(self.S), eng.dev(self.G)

    def run(self, iterations):
        assert hasattr(self, 'F') and hasattr(self, 'S') and hasattr(self, 'G'), \
            "F, S and G have not been initialised - please run NMTF.initialise() first."
        eng, F, S, G = self._state()
        self._start_run()
        pairs = list(itertools.product(range(0, self.K), range(0, self.L)))

        def body():
            eng.s_phase(F, S, G, pairs)               # reference order: S, F, G (nmtf_np.py:129-136)
            self._phase_F(eng, F, S, G)
            self._phase_G(eng, F, S, G)
            return _mm(F, S, False), G
        trace, secs = eng.run_loop(iterations, body)
        for it in range(iterations):
            self._record(trace[it], it + 1, secs[it])
        self.F, self.S, self.G = F.cpu().numpy(), S.cpu().numpy(), G.cpu().numpy()

    def train(self, iterations, init_S='random', init_FG='random', expo_prior=1.):
        self.initialise(init_S=init_S, init_FG=init_FG, expo_prior=expo_prior)
        self.run(iterations=iterations)

    def update_F(self, k):
        eng, F, S, G = self._state()
        self._phase_F(eng, F, S, G, single=k)
        self.F = F.cpu().numpy()

    def update_G(self, l):
        eng, F, S, G = self._state()
        self._phase_G(eng, F, S, G, single=l)
        self.G = G.cpu().numpy()

    def update_S(self, k, l):
        eng, F, S, G = self._state()
        eng.s_phase(F, S, G, [(k, l)])
        self.S = S.cpu().numpy()

    def triple_dot(self, M1, M2, M3):
        eng = self._engine()
        return self._mm(self._mm(eng.dev(M1), eng.dev(M2), False), eng.dev(M3), False).cpu().numpy()

    def _sums(self, M_pred=None):
        eng, F, S, G = self._state()
        return eng.sums(_mm(F, S, False), G, M_pred)

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums(M_pred))

    def compute_I_div(self):
        return float(self._sums()[7])

    def give_update(self, iteration):
        sums = self._sums()
        if not hasattr(self, 'all_performances'):
            self._start_run()
        self._record(sums, iteration, time.time())
