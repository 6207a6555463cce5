"""Drop-in classes for the reference's two-factor models, backed by the B200 engine.

    bnmf_gibbs_optimised  (code/models/bnmf_gibbs_optimised.py:53)
    bnmf_vb_optimised     (code/models/bnmf_vb_optimised.py:52)
    nmf_icm               (code/models/nmf_icm.py:46)

Same constructor arguments, method names, return values, attribute names and assertion messages as the
reference.  State attributes (U, V, tau, expU, muU, ...) are host numpy arrays, assignable as in the reference's
white-box tests; every method uploads them, runs CUDA kernels through the C ABI and downloads the result.
run(iterations) keeps the whole loop on the device (no host round trip per column or per iteration).
"""
import math

import numpy as np
import scipy.sparse
import torch

from . import _lib
from .data import validate_sparse
from .engine import Dataset, SparseDataset, engine_for, S_BETA_S, S_ELBO, S_ESD, S_LOGTAU, S_TAU, _ptr, _stream, require_cuda

def _elbo_alpha_s_correction(model):
    """The device evaluates the ELBO with alpha* = alpha + |Omega|/2, which is what update_tau() always yields.  The
    reference reads the ATTRIBUTE alpha_s instead (bnmf_vb_optimised.py:170, bnmtf_vb_optimised.py:217), and its
    white-box test assigns an arbitrary value (tests/code/test_bnmf_vb_optimised.py:183: alpha_s = 20): swap the three
    alpha*-dependent terms  -a log(beta*) + lgamma(a) - (a - 1) E[log tau]  on the host when the attribute differs."""
    a0 = model.alpha + model.size_Omega / 2.
    a = float(getattr(model, 'alpha_s', a0))
    if a == a0:
        return 0.
    b, elt = float(model.beta_s), float(model.explogtau)
    f = lambda x: -x * math.log(b) + math.lgamma(x) - (x - 1.) * elt
    return f(a) - f(a0)


# bytes moved host->device / device->host by the model classes of this process (bench.py's e2e block reports what one
# run(1) really copied, counted where the copies are issued)
XFER = [0, 0]



class _NoSharedHost(Exception):
    pass


class _LazySamples(object):
    """What bnmf_gibbs_optimised.run() returns: behaves like the reference's tuple (all_U, all_V, all_tau), but the two
    sample arrays are only downloaded from the device when somebody looks at them."""

    def __init__(self, model):
        self._m = model

    def __len__(self):
        return 3

    def __getitem__(self, i):
        return (self._m.all_U, self._m.all_V, self._m.all_tau)[i] if isinstance(i, slice) else \
            (self._m.all_U if i in (0, -3) else self._m.all_V if i in (1, -2) else self._m.all_tau if i in (2, -1) else
             (_ for _ in ()).throw(IndexError(i)))

    def __iter__(self):
        yield self._m.all_U
        yield self._m.all_V
        yield self._m.all_tau


def _shared_pinned(shape, register=True):
    """A float64 host array in POSIX shared memory, mapped and page-locked (cudaHostRegister) by every rank of the default
    process group: (torch view, numpy view, keep-alive).  Rank 0 creates the segment and unlinks it as soon as everybody
    has attached, so nothing is left behind in /dev/shm whatever happens to the processes."""
    import torch.distributed as dist
    from multiprocessing import resource_tracker, shared_memory
    nbytes = max(8, int(np.prod(shape)) * 8)
    rank = dist.get_rank()
    box = [None]
    shm = None
    if rank == 0:
        shm = shared_memory.SharedMemory(create=True, size=nbytes)
        box[0] = shm.name
    dist.broadcast_object_list(box, src=0)
    if rank != 0:
        shm = shared_memory.SharedMemory(name=box[0])
        try:                                             # attaching registered the segment with this process's tracker too
            resource_tracker.unregister(shm._name, "shared_memory")
        except Exception:
            pass
    dist.barrier()
    if rank == 0:
        shm.unlink()
    arr = np.ndarray(tuple(shape), dtype=np.float64, buffer=shm.buf)
    t = torch.from_numpy(arr)
    if register:
        ptr = t.data_ptr()
        rc = torch.cuda.cudart().cudaHostRegister(ptr, nbytes, 0)
        if int(rc) != 0:
            raise RuntimeError("cudaHostRegister failed (%s)" % rc)

        def _unregister(p=ptr):
            # before the mapping goes away: a later segment mapped at the same address could not be registered otherwise
            try:
                torch.cuda.cudart().cudaHostUnregister(p)
            except Exception:
                pass
        import weakref
        weakref.finalize(arr, _unregister)
    if rank == 0:
        arr[...] = 0.0
    dist.barrier()
    return t, arr, shm


def _shared_seed(seed, distributed):
    """Philox seed of a model: the caller's, else one derived from numpy's global state (_lib.derive_seed: distinct for
    successive models, reproducible after numpy.random.seed).  Sharded runs: rank 0's value is broadcast, so that the
    replicated tau draw and the row-keyed factor draws are the same stream on every rank whatever each rank's numpy
    state is."""
    seed = int(seed) if seed is not None else _lib.derive_seed()
    if distributed:
        import torch.distributed as dist
        if dist.is_initialized() and dist.get_world_size() > 1:
            box = [seed]
            dist.broadcast_object_list(box, src=0)
            seed = int(box[0])
    return seed


METRICS = ['MSE', 'R^2', 'Rp']
QUALITY = ['loglikelihood', 'BIC', 'AIC', 'MSE', 'ELBO']


def _metrics_from_sums(s):
    """{MSE,R^2,Rp} from the seven masked sums (e2, p, p2, rp, r, r2, n), reference :208-223."""
    e2, p, p2, rp, r, r2, n = (float(x) for x in s[:7])
    mean_r, mean_p = r / n, p / n
    ss_tot = r2 - r * mean_r
    with np.errstate(all='ignore'):
        R2 = 1. - e2 / ss_tot if ss_tot != 0. else np.inf
        Rp = np.float64(rp - r * mean_p) / (math.sqrt(max(ss_tot, 0.)) * math.sqrt(max(p2 - p * mean_p, 0.)))
    return {'MSE': e2 / n, 'R^2': R2, 'Rp': Rp}


class _TwoFactorBase(object):
    _mode = None

    def __init__(self, R, M, K, priors, device=None, seed=None, distributed=False):
        self._sparse = scipy.sparse.issparse(R)
        if self._sparse:
            # sparse input: the stored entries of R are its known entries (explicit zeros included), M (or None: all of
            # them) selects the training entries; self.R / self.M are canonical CSR matrices (data.validate_sparse)
            if distributed:
                raise ValueError("sparse R is not supported with distributed=True")
            self.R, self.M, self._train = validate_sparse(R, M)
            self.K = K
            (self.I, self.J) = self.R.shape
            self.size_Omega = float(self.M.nnz)
        else:
            self.R = np.array(R, dtype=float)
            self.M = np.array(M, dtype=float)
            self.K = K

            assert len(self.R.shape) == 2, "Input matrix R is not a two-dimensional array, " \
                "but instead %s-dimensional." % len(self.R.shape)
            assert self.R.shape == self.M.shape, "Input matrix R is not of the same size as " \
                "the indicator matrix M: %s and %s respectively." % (self.R.shape, self.M.shape)

            (self.I, self.J) = self.R.shape
            self.size_Omega = self.M.sum()
            self.check_empty_rows_columns()

        self.alpha, self.beta, self.lambdaU, self.lambdaV = \
            float(priors['alpha']), float(priors['beta']), np.array(priors['lambdaU']), np.array(priors['lambdaV'])
        if self.lambdaU.shape == ():
            self.lambdaU = self.lambdaU * np.ones((self.I, self.K))
        if self.lambdaV.shape == ():
            self.lambdaV = self.lambdaV * np.ones((self.J, self.K))

        assert self.lambdaU.shape == (self.I, self.K), "Prior matrix lambdaU has the wrong shape: %s instead of (%s, %s)." % (self.lambdaU.shape, self.I, self.K)
        assert self.lambdaV.shape == (self.J, self.K), "Prior matrix lambdaV has the wrong shape: %s instead of (%s, %s)." % (self.lambdaV.shape, self.J, self.K)

        self._device_arg, self._seed, self._eng = device, seed, None
        self._distributed = distributed   # True: shard rows of R / R^T over the ranks of torch.distributed
        self.verbose = False

    @classmethod
    def from_dataset(cls, dataset, K, priors, seed=None):
        """Build a model on an engine.Dataset that already lives on the GPU (matrices too large for, or never
        present in, host memory).  R and M stay None on the host; everything else behaves as usual."""
        self = cls.__new__(cls)
        self.R = self.M = None
        self.K = K
        (self.I, self.J) = (dataset.I, dataset.J)
        self.size_Omega = float(dataset.n_obs)
        self.alpha, self.beta = float(priors['alpha']), float(priors['beta'])
        self.lambdaU, self.lambdaV = np.array(priors['lambdaU'], dtype=float), np.array(priors['lambdaV'], dtype=float)
        if self.lambdaU.shape == ():
            self.lambdaU = self.lambdaU * np.ones((self.I, self.K))
        if self.lambdaV.shape == ():
            self.lambdaV = self.lambdaV * np.ones((self.J, self.K))
        self._device_arg, self._seed, self.verbose = dataset.device, seed, False
        self._distributed = dataset.world > 1
        self._eng = engine_for(dataset, K, cls._mode, self.alpha, self.beta, seed=_shared_seed(seed, dataset.world > 1))
        return self

    def check_empty_rows_columns(self):
        sums_columns = self.M.sum(axis=0)
        sums_rows = self.M.sum(axis=1)
        for i, c in enumerate(sums_rows):
            assert c != 0, "Fully unobserved row in R, row %s." % i
        for j, c in enumerate(sums_columns):
            assert c != 0, "Fully unobserved column in R, column %s." % j

    # ---- device plumbing --------------------------------------------------------------------------------
    def _engine(self):
        if self._eng is None:
            dev = require_cuda(self._device_arg)
            world, rank = 1, 0
            if self._distributed:
                import torch.distributed as dist
                world, rank = dist.get_world_size(), dist.get_rank()
            if self._sparse:
                ds = SparseDataset(self.R, self._train, dev)
            else:
                ds = Dataset.from_host(self.R, self.M, dev, world, rank)
            self._eng = engine_for(ds, self.K, self._mode, self.alpha, self.beta,
                                   seed=_shared_seed(self._seed, self._distributed))
        return self._eng

    @staticmethod
    def _up(dst, src):
        src = np.ascontiguousarray(src, dtype=np.float64)
        XFER[0] += src.nbytes
        dst[:src.shape[0]].copy_(torch.from_numpy(src), non_blocking=False)

    @staticmethod
    def _down(src, n=None):
        t = (src if n is None else src[:n]).detach()
        XFER[1] += t.numel() * t.element_size()
        return t.cpu().numpy().copy()

    def _xfer_bytes(self):
        """(host->device, device->host) bytes of the last run() of this model."""
        return getattr(self, '_last_xfer', (0, 0))

    def _xfer_mark(self, start=None):
        if start is None:
            return (XFER[0], XFER[1])
        self._last_xfer = (XFER[0] - start[0], XFER[1] - start[1])

    # Factor state crosses PCIe through persistent page-locked buffers.  After run() the state attributes (U, expU, ...)
    # ARE numpy views of those buffers, rewritten in place by the next run() -- the same aliasing the reference has,
    # whose updates write into self.U in place -- and _push() DMAs straight from them (no staging copy) as long as
    # the attribute still is that view; anything the caller assigned instead takes the pageable path.
    #
    # Row-sharded runs (one process per GPU of one node): the buffers live in POSIX shared memory mapped -- and
    # page-locked -- by every rank, so that each rank moves only ITS OWN rows of the factor state over its PCIe link
    # (upload: own rows, then peer stores replicate them to the other GPUs over NVLink; download: own rows into the
    # shared array) and every rank still ends up with the complete host arrays, as the reference's attributes are.
    def _own_rows(self, f):
        """(sharded-with-shared-host-buffers?, lo, cnt) for the rows of Factor f this rank moves."""
        eng = self._eng
        if eng is not None and eng.comm.world > 1 and eng.comm.sync is not None and f.peer is not None \
                and not self.__dict__.get('_no_shared_host', False):
            return True, f.part.lo(), f.part.cnt()
        return False, 0, f.n

    def _host_buffer(self, key, shape, shared):
        pins = self.__dict__.setdefault('_pins', {})
        ent = pins.get(key)
        if ent is not None and tuple(ent[0].shape) == tuple(shape) and ent[2] == shared:
            return ent
        if shared:
            try:
                t, arr, shm = _shared_pinned(shape)
                ent = pins[key] = (t, arr, True, shm)
                return ent
            except Exception as exc:                      # no /dev/shm, registration refused, ...: private buffers, full copies
                import warnings
                warnings.warn("bnmtf_b200: shared page-locked host buffers unavailable (%s: %s); every rank moves the "
                              "whole factor state" % (type(exc).__name__, exc))
                self._no_shared_host = True
                raise _NoSharedHost()
        buf = torch.empty(tuple(shape), dtype=torch.float64, pin_memory=True)
        ent = pins[key] = (buf, buf.numpy(), False, None)
        return ent

    def _down_s(self, key, src, f):
        shared, lo, cnt = self._own_rows(f)
        try:
            ent = self._host_buffer(key, (f.n,) + tuple(src.shape[1:]), shared)
        except _NoSharedHost:
            shared, lo, cnt = False, 0, f.n
            ent = self._host_buffer(key, (f.n,) + tuple(src.shape[1:]), False)
        if cnt > 0:
            t = src[lo:lo + cnt]
            XFER[1] += t.numel() * t.element_size()
            ent[0][lo:lo + cnt].copy_(t, non_blocking=True)       # _pull_done() synchronises before the views are read
        return ent[1]

    def _pull_done(self, eng):
        """All device->host copies of this run have landed -- on every rank, when the host buffers are shared."""
        if eng.comm.world > 1 and eng.comm.sync is not None and not self.__dict__.get('_no_shared_host', False):
            eng.comm.barrier(3)      # a rank's barrier kernel runs after its copies on the stream: when ours has finished, all have
        torch.cuda.current_stream().synchronize()

    def _up_s(self, key, dst, src, f=None, replicate=True):
        """Host state -> device.  f given and the run is sharded: only this rank's rows cross PCIe; replicate: the other
        ranks' copies are completed over NVLink (needed for the factors themselves, not for mu / tau / lambda, of which a
        rank only reads its own rows).  Returns True if a cross-GPU barrier has to follow (_push_done)."""
        ent = self.__dict__.get('_pins', {}).get(key)
        shared, lo, cnt = self._own_rows(f) if f is not None else (False, 0, src.shape[0])
        if shared:
            if cnt > 0:
                if ent is not None and src is ent[1]:
                    XFER[0] += cnt * int(np.prod(src.shape[1:])) * 8
                    dst[lo:lo + cnt].copy_(ent[0][lo:lo + cnt], non_blocking=True)
                else:
                    rows = np.ascontiguousarray(src[lo:lo + cnt], dtype=np.float64)
                    XFER[0] += rows.nbytes
                    dst[lo:lo + cnt].copy_(torch.from_numpy(rows), non_blocking=False)
            if replicate:
                peers = f.peer[1] if dst is f.fac else f.peer[2]
                self._eng.comm.put_rows(dst, f.part, peers)
                self._need_barrier = True
            return
        if ent is not None and src is ent[1]:
            XFER[0] += src.nbytes
            dst[:src.shape[0]].copy_(ent[0], non_blocking=True)
        else:
            self._up(dst, src)

    def _up_lam(self, key, f, value):
        """The priors do not change between run() calls: uploaded when the attribute is a different object than last time."""
        sent = self.__dict__.setdefault('_lam_sent', {})
        if sent.get(key) is value:
            return
        shared, lo, cnt = self._own_rows(f)
        if shared:
            if cnt > 0:
                rows = np.ascontiguousarray(value[lo:lo + cnt], dtype=np.float64)
                XFER[0] += rows.nbytes
                f.lam[lo:lo + cnt].copy_(torch.from_numpy(rows))
        else:
            self._up(f.lam, value)
        sent[key] = value

    def _push_done(self, eng):
        if self.__dict__.pop('_need_barrier', False):
            eng.comm.barrier(3)      # every rank's rows are in every copy before the first kernel reads a factor

    def _set_scalars(self, eng, kv):
        idx = torch.tensor(list(kv.keys()), dtype=torch.int64)
        val = torch.tensor([float(v) for v in kv.values()], dtype=torch.float64)
        eng.scalars.index_copy_(0, idx.to(eng.scalars.device), val.to(eng.scalars.device))

    def _sums_for(self, M_pred, U, V):
        """Seven masked sums of the prediction U V^T over M_pred, on the device."""
        eng = self._engine()
        self._up(eng.U.fac, U)
        self._up(eng.V.fac, V)
        bits = eng.ds.bits if M_pred is None else eng.ds.pack_mask(M_pred)
        eng.metrics(bits)
        return eng.m8.cpu().numpy()

    # ---- metric helpers on explicit matrices (reference :208-223) ----------------------------------------------
    def _dense_sums(self, M, R, R_pred):
        dev = require_cuda(self._device_arg)
        t = [torch.from_numpy(np.ascontiguousarray(np.broadcast_to(x, np.shape(R)), dtype=np.float64)).to(dev) for x in (R, R_pred, M)]
        nb = 64
        part = torch.zeros(nb * 8, dtype=torch.float64, device=dev)
        out = torch.zeros(8, dtype=torch.float64, device=dev)
        _lib.call("bnmtf_dense_metrics_f64", _ptr(t[0]), _ptr(t[1]), _ptr(t[2]), t[0].numel(), _ptr(part), nb, _ptr(out), _stream())
        return out.cpu().numpy()

    def compute_MSE(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['MSE']

    def compute_R2(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['R^2']

    def compute_Rp(self, M, R, R_pred):
        return _metrics_from_sums(self._dense_sums(M, R, R_pred))['Rp']

    def _n_params(self):
        return self.I * self.K + self.J * self.K

    def _quality_from_ll(self, metric, log_likelihood):
        if metric == 'loglikelihood':
            return log_likelihood
        elif metric == 'BIC':
            return - 2 * log_likelihood + self._n_params() * math.log(self.size_Omega)
        elif metric == 'AIC':
            return - 2 * log_likelihood + 2 * self._n_params()

    def _init_trace_lists(self):
        self.all_times = []
        self.all_performances = {}
        for metric in METRICS:
            self.all_performances[metric] = []

    def _run_loop(self, eng, iterations, minimum_TN=0.0, per_iteration=None, samples=None, sums=None):
        """Enqueue `iterations` sweeps; CUDA events give the reference's cumulative all_times.  samples = (all_U, all_V):
        device tensors for the draw of every sweep, filled by per_iteration -- or by the kernel itself when the problem is
        small enough for the single-kernel sweep (csrc/small.cu: the whole run is then one launch, and all_times comes
        from the device's own clock)."""
        eng.alloc_trace(iterations)
        launched = False
        if iterations > 0 and eng.small_cluster() and (per_iteration is None or samples is not None or sums is not None):
            times = torch.zeros(iterations + 1, dtype=torch.int64, device=eng.ds.device)
            try:
                eng.sweep_many(iterations, minimum_TN, samples, times, sums)
                launched = True
            except _lib.BnmtfError as exc:
                # e.g. no 16 free SMs in one GPC for the cluster while other work runs: nothing has been modified, the
                # multi-kernel path below does the same run
                import warnings
                warnings.warn("bnmtf_b200: single-kernel sweep not launched (%s); using the per-phase kernels" % exc)
                eng._small_c = 0
        if launched:
            torch.cuda.synchronize()
            t = times.cpu().numpy()
            self.all_times = [float(x - t[0]) / 1e9 for x in t[1:]]
            XFER[1] += iterations * 64
            tr = eng.trace[:iterations].cpu().numpy()
            for i, metric in enumerate(METRICS):
                self.all_performances[metric] = [float(v) for v in tr[:, 1 + i]]
            return tr
        start = torch.cuda.Event(enable_timing=True)
        marks = []
        start.record()
        for it in range(iterations):
            eng.sweep(minimum_TN)
            if per_iteration is not None:
                per_iteration(it)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
        torch.cuda.synchronize()
        self.all_times = [start.elapsed_time(ev) / 1e3 for ev in marks]
        XFER[1] += iterations * 64
        tr = eng.trace[:iterations].cpu().numpy()
        for i, metric in enumerate(METRICS):
            self.all_performances[metric] = [float(v) for v in tr[:, 1 + i]]
        return tr


# =====================================================================================================
class bnmf_gibbs_optimised(_TwoFactorBase):
    """Gibbs sampler for BNMF (reference code/models/bnmf_gibbs_optimised.py)."""
    _mode = 'gibbs'

    def train(self, init, iterations):
        self.initialise(init=init)
        return self.run(iterations)

    def initialise(self, init='random'):
        assert init in ['random', 'exp'], "Unknown initialisation option: %s. Should be 'random' or 'exp'." % init
        if init == 'random':
            # same numpy stream order as the reference's (i,k) then (j,k) loops (:106-109)
            self.U = np.random.exponential(scale=1.0 / self.lambdaU)
            self.V = np.random.exponential(scale=1.0 / self.lambdaV)
        else:
            self.U, self.V = 1.0 / self.lambdaU, 1.0 / self.lambdaV
        self.tau = self.alpha_s() / self.beta_s()

    def _push(self):
        eng = self._engine()
        self._up_s('U', eng.U.fac, self.U, eng.U), self._up_s('V', eng.V.fac, self.V, eng.V)
        self._up_lam('lambdaU', eng.U, self.lambdaU), self._up_lam('lambdaV', eng.V, self.lambdaV)
        self._set_scalars(eng, {S_TAU: float(getattr(self, 'tau', 1.0))})
        self._push_done(eng)
        return eng

    def run(self, iterations, summary=None):
        """The reference's run(iterations).  The draws of every iteration stay ON THE DEVICE (each rank keeps its own rows):
        all_U / all_V are downloaded the first time somebody reads them (or the returned tuple), approx_expectation /
        predict / quality average them on the device.

        summary=(burn_in, thinning): keep only the running sums over range(burn_in, iterations, thinning) -- what
        approx_expectation(burn_in, thinning) needs -- instead of iterations x (I + J) x K samples; all_U / all_V are then
        not available.  This is how a long chain on a matrix of the benchmark's size is run (1000 iterations at
        65536 x 32768, K=20 would be 15.7 GB of samples)."""
        x0 = self._xfer_mark()
        eng = self._push()
        dev = eng.ds.device
        lo_u, n_u, lo_v, n_v = eng.loc[0][0], eng.loc[0][1], eng.loc[1][0], eng.loc[1][1]
        self._samples = None
        for key in ('_all_U', '_all_V', '_cache_U', '_cache_V'):
            self.__dict__.pop(key, None)
        if summary is not None:
            burn_in, thinning = int(summary[0]), int(summary[1])
            assert thinning >= 1 and 0 <= burn_in < max(1, iterations), "summary=(burn_in, thinning) selects no iteration"
            keepers = set(range(burn_in, iterations, thinning))
            sums = (torch.zeros((max(n_u, 1), self.K), dtype=torch.float64, device=dev),
                    torch.zeros((max(n_v, 1), self.K), dtype=torch.float64, device=dev))
            store = {'kind': 'sums', 'window': (burn_in, thinning), 'count': len(keepers), 'U': sums[0], 'V': sums[1]}

            def keep(it):
                if it in keepers:
                    if n_u:
                        _lib.call("bnmtf_accumulate_f64", _ptr(sums[0]), _ptr(eng.U.fac, lo_u), n_u * self.K, _stream())
                    if n_v:
                        _lib.call("bnmtf_accumulate_f64", _ptr(sums[1]), _ptr(eng.V.fac, lo_v), n_v * self.K, _stream())
        else:
            need = iterations * (n_u + n_v) * self.K * 8
            # (cudaMemGetInfo costs milliseconds: only asked when the draws are sizeable)
            free = torch.cuda.mem_get_info(dev)[0] if need > (1 << 28) else float("inf")
            if need > 0.8 * free:
                raise _lib.BnmtfError("run(%d) would keep %.1f GB of samples on the device (%.1f GB free): pass "
                                      "summary=(burn_in, thinning) to keep running sums instead" % (iterations, need / 1e9, free / 1e9))
            all_U = torch.zeros((iterations, max(n_u, 1), self.K), dtype=torch.float64, device=dev)
            all_V = torch.zeros((iterations, max(n_v, 1), self.K), dtype=torch.float64, device=dev)
            store = {'kind': 'all', 'U': all_U, 'V': all_V}

            def keep(it):
                # own rows only: nobody else writes them, so a faster peer's next sweep cannot interleave with this copy
                if n_u:
                    all_U[it, :n_u].copy_(eng.U.fac[lo_u:lo_u + n_u])
                if n_v:
                    all_V[it, :n_v].copy_(eng.V.fac[lo_v:lo_v + n_v])
        self._init_trace_lists()
        tr = self._run_loop(eng, iterations, per_iteration=keep, samples=(all_U, all_V) if summary is None else None,
                            sums=(sums[0], sums[1], burn_in, thinning) if summary is not None else None)
        store['iterations'] = iterations
        self._samples = store
        self.U, self.V = self._down_s('U', eng.U.fac, eng.U), self._down_s('V', eng.V.fac, eng.V)
        self._pull_done(eng)
        self.all_tau = tr[:, 0].copy()
        if iterations > 0:
            self.tau = float(tr[-1, 0])
        if self.verbose:
            for it in range(iterations):
                print("Iteration %s. MSE: %s. R^2: %s. Rp: %s." % (it + 1, tr[it, 1], tr[it, 2], tr[it, 3]))
        self._xfer_mark(x0)
        return _LazySamples(self)

    # all_U / all_V: host copies of the device-resident draws, made on first access; assignable as in the reference's tests
    def _materialise(self, which):
        if '_all_' + which in self.__dict__:              # assigned by the caller
            return self.__dict__['_all_' + which]
        cache = self.__dict__.get('_cache_' + which)
        if cache is not None:
            return cache
        st = self.__dict__.get('_samples')
        if st is None:
            raise AttributeError("all_%s: no samples yet (call run())" % which)
        if st['kind'] != 'all':
            raise AttributeError("all_%s was not kept: run(..., summary=%r) stores running sums only" % (which, st['window']))
        eng = self._engine()
        f = eng.U if which == 'U' else eng.V
        lo, cnt = eng.loc[0 if which == 'U' else 1]
        its = st['iterations']
        if eng.comm.world > 1:
            # every rank holds its own rows of every draw: all-gather them per draw into the replicated layout
            full = torch.zeros((its, f.part.n_pad, self.K), dtype=torch.float64, device=eng.ds.device)
            if cnt:
                full[:, lo:lo + cnt] = st[which][:, :cnt]
            for it in range(its):
                eng.comm.gather_rows(full[it], f.part)
            host = self._down(full[:, :f.n])
        else:
            host = self._down(st[which][:, :f.n])
        self.__dict__['_cache_' + which] = host
        return host

    all_U = property(lambda self: self._materialise('U'), lambda self, v: self.__dict__.__setitem__('_all_U', v))
    all_V = property(lambda self: self._materialise('V'), lambda self, v: self.__dict__.__setitem__('_all_V', v))

    # ---- conditional parameters (reference :161-177) -----------------------------------------------------
    def alpha_s(self):
        return self.alpha + self.size_Omega / 2.0

    def beta_s(self):
        return self.beta + 0.5 * float(self._sums_for(None, self.U, self.V)[0])

    def _params(self, side, k):
        eng = self._push()
        eng.stats(side)
        eng.solve(side, order=[k], apply=False, want_sterm=True, use_iter=False)
        me = eng.U if side == 0 else eng.V
        eng.gather_params()
        return self._down(me.tauf, me.n)[:, k], self._down(eng.sterm, me.n)[:, k]

    def tauU(self, k):
        return self._params(0, k)[0]

    def muU(self, tauUk, k):
        s = self._params(0, k)[1]
        with np.errstate(all='ignore'):
            return 1. / np.asarray(tauUk) * (-self.lambdaU[:, k] + self.tau * s)

    def tauV(self, k):
        return self._params(1, k)[0]

    def muV(self, tauVk, k):
        s = self._params(1, k)[1]
        with np.errstate(all='ignore'):
            return 1. / np.asarray(tauVk) * (-self.lambdaV[:, k] + self.tau * s)

    # ---- posterior summaries (reference :182-251) -------------------------------------------------------------
    def approx_expectation(self, burn_in, thinning):
        """Posterior means over range(burn_in, iterations, thinning) (reference :182-187), averaged on the device from the
        device-resident draws or running sums; draws assigned by the caller as host arrays are uploaded first."""
        st = self.__dict__.get('_samples')
        own_host = '_all_U' in self.__dict__ or st is None          # draws assigned by the caller as host arrays
        indices = range(burn_in, len(self.all_U) if own_host else st['iterations'], thinning)
        n = float(len(indices))
        exp_tau = sum([self.all_tau[i] for i in indices]) / n
        eng = self._engine()
        dev = eng.ds.device
        if own_host:
            out = []
            for a in (self.all_U, self.all_V):
                a = np.ascontiguousarray(a, dtype=np.float64)
                d = torch.from_numpy(a).to(dev)
                o = torch.zeros(a.shape[1:], dtype=torch.float64, device=dev)
                _lib.call("bnmtf_sample_mean_f64", _ptr(d), int(np.prod(a.shape[1:])), a.shape[0], burn_in, thinning, _ptr(o), _stream())
                out.append(self._down(o))
            return (out[0], out[1], exp_tau)
        out = []
        for which, f, side in (('U', eng.U, 0), ('V', eng.V, 1)):
            lo, cnt = eng.loc[side]
            full = torch.zeros((f.part.n_pad, self.K), dtype=torch.float64, device=dev)
            if cnt:
                if st['kind'] == 'sums':
                    assert (burn_in, thinning) == st['window'], \
                        "this chain kept running sums for (burn_in, thinning) = %r only" % (st['window'],)
                    full[lo:lo + cnt] = st[which][:cnt]            # the sums; divided by the count on the host below
                else:
                    dense = st[which] if st[which].shape[1] == cnt else st[which][:, :cnt].contiguous()
                    tmp = torch.zeros((cnt, self.K), dtype=torch.float64, device=dev)
                    _lib.call("bnmtf_sample_mean_f64", _ptr(dense), cnt * self.K, st['iterations'], burn_in, thinning, _ptr(tmp), _stream())
                    full[lo:lo + cnt] = tmp
            eng.comm.gather_rows(full, f.part)
            host = self._down(full, f.n)
            out.append(host / float(st['count']) if st['kind'] == 'sums' else host)
        return (out[0], out[1], exp_tau)

    def predict(self, M_pred, burn_in, thinning):
        (exp_U, exp_V, _) = self.approx_expectation(burn_in, thinning)
        return _metrics_from_sums(self._sums_for(M_pred, exp_U, exp_V))

    def predict_while_running(self):
        return _metrics_from_sums(self._sums_for(None, self.U, self.V))

    def quality(self, metric, burn_in, thinning):
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        (expU, expV, exptau) = self.approx_expectation(burn_in, thinning)
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, expU, expV))['MSE']
        elif metric == 'ELBO':
            return 0.
        return self._quality_from_ll(metric, self.log_likelihood(expU, expV, exptau))

    def log_likelihood(self, expU, expV, exptau):
        explogtau = math.log(exptau)
        return self.size_Omega / 2. * (explogtau - math.log(2 * math.pi)) \
            - exptau / 2. * float(self._sums_for(None, expU, expV)[0])


# =====================================================================================================
class nmf_icm(_TwoFactorBase):
    """Iterated conditional modes (MAP) for NMF (reference code/models/nmf_icm.py)."""
    _mode = 'icm'

    def train(self, init, iterations):
        self.initialise(init=init)
        return self.run(iterations)

    def initialise(self, init='random'):
        assert init in ['random', 'exp'], "Unknown initialisation option: %s. Should be 'random' or 'exp'." % init
        if init == 'random':
            self.U = np.random.exponential(scale=1.0 / self.lambdaU)
            self.V = np.random.exponential(scale=1.0 / self.lambdaV)
        else:
            self.U, self.V = 1.0 / self.lambdaU, 1.0 / self.lambdaV
        self.tau = (self.alpha_s() - 1.) / self.beta_s()

    _push = bnmf_gibbs_optimised._push
    alpha_s = bnmf_gibbs_optimised.alpha_s
    beta_s = bnmf_gibbs_optimised.beta_s
    _params = bnmf_gibbs_optimised._params
    tauU, muU, tauV, muV = (bnmf_gibbs_optimised.tauU, bnmf_gibbs_optimised.muU,
                            bnmf_gibbs_optimised.tauV, bnmf_gibbs_optimised.muV)

    def run(self, iterations, minimum_TN=0.):
        x0 = self._xfer_mark()
        eng = self._push()
        self._init_trace_lists()
        tr = self._run_loop(eng, iterations, minimum_TN=minimum_TN)
        self.all_tau = tr[:, 0].copy()
        self.U, self.V = self._down_s('U', eng.U.fac, eng.U), self._down_s('V', eng.V.fac, eng.V)
        self._pull_done(eng)
        if iterations > 0:
            self.tau = float(tr[-1, 0])
        self._xfer_mark(x0)
        return

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums_for(M_pred, self.U, self.V))

    def quality(self, metric):
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, self.U, self.V))['MSE']
        elif metric == 'ELBO':
            return 0.
        return self._quality_from_ll(metric, self.log_likelihood())

    def log_likelihood(self):
        return self.size_Omega / 2. * (math.log(self.tau) - math.log(2 * math.pi)) \
            - self.tau / 2. * float(self._sums_for(None, self.U, self.V)[0])


# =====================================================================================================
class bnmf_vb_optimised(_TwoFactorBase):
    """Variational Bayes for BNMF (reference code/models/bnmf_vb_optimised.py)."""
    _mode = 'vb'
    _STATE = ('expU', 'varU', 'muU', 'tauU', 'expV', 'varV', 'muV', 'tauV')

    def initialise(self, init='exp', tauUV={}):
        self.tauU = tauUV['tauU'] if 'tauU' in tauUV else np.ones((self.I, self.K))
        self.tauV = tauUV['tauV'] if 'tauV' in tauUV else np.ones((self.J, self.K))
        assert init in ['exp', 'random'], "Unrecognised init option for F,G: %s." % init
        self.muU, self.muV = 1. / self.lambdaU, 1. / self.lambdaV
        if init == 'random':
            self.muU = np.random.exponential(scale=1.0 / self.lambdaU)
            self.muV = np.random.exponential(scale=1.0 / self.lambdaV)
        # (the reference's column-by-column update_exp_U / update_exp_V loops, :112-115, as one device call per factor: the
        # moments are element-wise)
        from .distributions import TN_matrix_moments
        self.expU, self.varU = TN_matrix_moments(self.muU, self.tauU)
        self.expV, self.varV = TN_matrix_moments(self.muV, self.tauV)
        self.update_tau()
        self.update_exp_tau()

    def train(self, iterations, init_UV='random'):
        self.initialise(init=init_UV)      # the reference passes init_UV= to a signature without it (:157-159)
        self.run(iterations=iterations)

    def _push(self):
        eng = self._engine()
        for f, s in ((eng.U, 'U'), (eng.V, 'V')):
            # attributes the caller has not set yet are simply not uploaded: the reference's white-box tests call
            # exp_square_diff() / update_tau() / elbo() on objects that only carry the attributes those formulas read
            for attr, t in (('exp', f.fac), ('var', f.var), ('mu', f.mu), ('tau', f.tauf)):
                value = getattr(self, attr + s, None)
                if value is not None:
                    self._up_s(attr + s, t, value, f, replicate=attr in ('exp', 'var'))
            self._up_lam('lambda' + s, f, getattr(self, 'lambda' + s))
        self._set_scalars(eng, {S_TAU: float(getattr(self, 'exptau', 1.0)), S_LOGTAU: float(getattr(self, 'explogtau', 0.0)),
                                  S_BETA_S: float(getattr(self, 'beta_s', 1.0))})
        self._push_done(eng)
        return eng

    def _pull(self, eng, names=None):
        if not self._own_rows(eng.U)[0]:
            eng.gather_params()          # mu / tau of the other ranks' rows (with shared host buffers each rank writes its own)
        for f, s in ((eng.U, 'U'), (eng.V, 'V')):
            for attr, t in (('exp', f.fac), ('var', f.var), ('mu', f.mu), ('tau', f.tauf)):
                if names is None or attr + s in names:
                    setattr(self, attr + s, self._down_s(attr + s, t, f))
        self._pull_done(eng)

    def run(self, iterations):
        x0 = self._xfer_mark()
        eng = self._push()
        self._init_trace_lists()
        tr = self._run_loop(eng, iterations)
        self.all_exp_tau = [float(v) for v in tr[:, 0]]
        self.all_elbo = [float(v) for v in tr[:, 4]]
        self._pull(eng)
        if iterations > 0:
            sc = eng.scalars.cpu().numpy()
            self.exptau, self.explogtau = float(sc[S_TAU]), float(sc[S_LOGTAU])
            self.alpha_s, self.beta_s = self.alpha + self.size_Omega / 2.0, float(sc[S_BETA_S])
        if self.verbose:
            for it in range(iterations):
                print("Iteration %s. ELBO: %s. MSE: %s. R^2: %s. Rp: %s." % (it + 1, tr[it, 4], tr[it, 1], tr[it, 2], tr[it, 3]))
        self._xfer_mark(x0)
        return

    # ---- white-box pieces (reference :163-215) ---------------------------------------------------------------
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

    def _update_params(self, side, k):
        eng = self._push()
        eng.stats(side)
        eng.solve(side, order=[k], apply=False, use_iter=False)
        s = 'U' if side == 0 else 'V'
        f = eng.U if side == 0 else eng.V
        getattr(self, 'tau' + s)[:, k] = self._down(f.tauf, f.n)[:, k]
        getattr(self, 'mu' + s)[:, k] = self._down(f.mu, f.n)[:, k]

    def update_U(self, k):
        self._update_params(0, k)

    def update_V(self, k):
        self._update_params(1, k)

    def _update_exp(self, s, k):
        from .distributions import TN_vector_expectation, TN_vector_variance
        mu, tau = getattr(self, 'mu' + s)[:, k], getattr(self, 'tau' + s)[:, k]
        getattr(self, 'exp' + s)[:, k] = TN_vector_expectation(mu, tau)
        getattr(self, 'var' + s)[:, k] = TN_vector_variance(mu, tau)

    def update_exp_U(self, k):
        self._update_exp('U', k)

    def update_exp_V(self, k):
        self._update_exp('V', k)

    def predict(self, M_pred):
        return _metrics_from_sums(self._sums_for(M_pred, self.expU, self.expV))

    def quality(self, metric):
        metric = 'ELBO' if metric == 'elbo' else metric      # BASELINE.json spells it lower case
        assert metric in QUALITY, 'Unrecognised metric for model quality: %s.' % metric
        if metric == 'MSE':
            return _metrics_from_sums(self._sums_for(None, self.expU, self.expV))['MSE']
        elif metric == 'ELBO':
            return self.elbo()
        return self._quality_from_ll(metric, self.log_likelihood())

    def log_likelihood(self):
        return self.size_Omega / 2. * (self.explogtau - math.log(2 * math.pi)) \
            - self.exptau / 2. * float(self._sums_for(None, self.expU, self.expV)[0])


# BASELINE.json's names for the same classes
BNMF_Gibbs = bnmf_gibbs_optimised
BNMF_VB = bnmf_vb_optimised
