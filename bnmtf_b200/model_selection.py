"""Model selection and cross-validation drivers (the callers of the hot path: SURVEY.md section 8f, item 1).

Same classes, constructor arguments, methods, result attributes and log-file lines as the reference's
code/cross_validation/{line_search_bnmf, grid_search_bnmtf, greedy_search_bnmtf, line_search_cross_validation,
greedy_search_cross_validation, matrix_cross_validation, parallel_matrix_cross_validation,
nested_matrix_cross_validation}.py, so scripts written against those modules only change their import.  The
`classifier` / `method` argument is any class with the duck-typed model protocol (SURVEY.md 8b) -- normally the GPU
model classes of this package.

What is different is how the independent fits are executed.  The reference runs every (K[, L]) point, restart and fold
one after the other (or, for ParallelMatrixCrossValidation, in a multiprocessing.Pool of CPU workers).  Here a
`DevicePool` hands the fits to the GPUs of the box, one worker thread per GPU (BASELINE.json, config 5: "folds x grid
points across 8 B200").  With one GPU -- or `devices=1` -- the fits run inline in exactly the reference's order, so the
host random streams (numpy for the initialisations, python's `random` for folds, K-means and the VB-NMTF update order)
are consumed identically and seeded runs reproduce the reference's numbers (tests/test_model_selection.py).  With
several GPUs the candidate models are still built and initialised in that order, but they run concurrently: models
that draw host random numbers inside run() are then no longer bit-reproducible.

Deliberately kept quirks of the reference (file:line in the methods below): GreedySearchCrossValidation searches on the
FULL mask, not on the training fold; GreedySearch's K-only tail stores the last L-direction score as the running best.
"""
import json
import os
import threading

import numpy as np

from . import mask

metrics = ['BIC', 'AIC', 'loglikelihood', 'MSE', 'ELBO']
measures = ['R^2', 'MSE', 'Rp']
attempts_generate_M = 1000


# ---------------------------------------------------------------------------------------------------------------
class DevicePool:
    """Runs independent jobs on the GPUs of this box: one worker thread per device, each inside
    `torch.cuda.device(i)` (the model classes create their engine on the current device).  The GIL is released during
    kernel launches (ctypes) and synchronisation, so the devices work concurrently.  devices: None = all visible
    GPUs, an int = that many, a list = those device indices.  One device (or none visible): jobs run inline, in order."""

    def __init__(self, devices=None):
        try:
            import torch
            n = torch.cuda.device_count() if torch.cuda.is_available() else 0
        except Exception:
            n = 0
        if devices is None and os.environ.get("BNMTF_SELECTION_DEVICES"):
            devices = int(os.environ["BNMTF_SELECTION_DEVICES"])
        if devices is None:
            self.devices = list(range(n))
        elif isinstance(devices, int):
            self.devices = list(range(min(devices, n))) if n else []
        else:
            self.devices = list(devices)

    def device_for(self, i):
        """Device of job number i (static round-robin, so that a job's model can be built on its device beforehand)."""
        return self.devices[i % len(self.devices)] if self.devices else None

    def on(self, i):
        """Context manager: make device_for(i) the calling thread's current CUDA device.  Uses set_device, not the
        torch.cuda.device() guard: the guard defers cudaSetDevice until torch itself issues a CUDA call, but the
        kernels of this package are launched through ctypes on the runtime's current device."""
        import contextlib
        dev = self.device_for(i)
        if dev is None or len(self.devices) <= 1:
            return contextlib.nullcontext()
        import torch

        @contextlib.contextmanager
        def guard():
            prev = torch.cuda.current_device()
            torch.cuda.set_device(dev)
            try:
                yield
            finally:
                torch.cuda.set_device(prev)
        return guard()

    def map(self, fn, jobs):
        """[fn(job) for job in jobs]; job i runs on device_for(i), the jobs of one device in order on one thread.  The
        first exception is re-raised."""
        jobs = list(jobs)
        if len(self.devices) <= 1 or len(jobs) <= 1:
            return [fn(j) for j in jobs]
        import torch
        from . import engine
        results, errors = [None] * len(jobs), []

        def worker(slot):
            torch.cuda.set_device(self.devices[slot])
            torch.empty(1, device="cuda:%d" % self.devices[slot])      # make sure the context exists
            engine.thread_flags.no_graph = True
            for i in range(slot, len(jobs), len(self.devices)):
                if errors:
                    return
                try:
                    results[i] = fn(jobs[i])
                except BaseException as e:   # noqa: B902 -- reported to the caller below
                    errors.append(e)
                    return
        threads = [threading.Thread(target=worker, args=(s,)) for s in range(min(len(self.devices), len(jobs)))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return results


def _pin_seed(model):
    """Models of this package draw their Philox seed from numpy's stream when the engine is first created; do it now,
    on the calling thread, so that concurrent runs stay reproducible."""
    if getattr(model, '_seed', 0) is None and getattr(model, '_eng', 0) is None:
        from . import _lib
        model._seed = _lib.derive_seed()


def _home(model):
    """Context manager: the CUDA device a model of this package lives on (its kernels are launched on the calling
    thread's current device); a no-op for foreign classifiers and for models that have not touched a device yet."""
    import contextlib
    eng = getattr(model, '_eng', None)
    dev = getattr(getattr(eng, 'ds', None), 'device', None) if eng is not None else None
    if dev is None:
        return contextlib.nullcontext()
    import torch

    @contextlib.contextmanager
    def home():
        prev = torch.cuda.current_device()
        torch.cuda.set_device(dev)       # eager cudaSetDevice (see DevicePool.map)
        try:
            yield
        finally:
            torch.cuda.set_device(prev)
    return home()


def _quality_args(burn_in, thinning):
    return (burn_in, thinning) if burn_in is not None and thinning is not None else ()


# ---- sparse input (DESIGN.md section 12) ------------------------------------------------------------------------
class _Entries:
    """A training set of sparse input: R's canonical CSR `Rc` and a bool per stored entry of it (`train`).  The fits of
    this package's model classes on it are built with from_dataset on one shared engine.SparseDataset per CUDA device,
    made on first use and dropped by release(); any other classifier gets its constructor with (Rc, a CSR mask)."""

    def __init__(self, Rc, train):
        self.Rc, self.train = Rc, train
        self._ds, self._mask = {}, None

    def mask(self):
        if self._mask is None:
            self._mask = mask._entry_mask(self.Rc, self.train)
        return self._mask

    def dataset(self):
        """The SparseDataset of these entries on the calling thread's current device."""
        from .engine import SparseDataset, require_cuda
        dev = require_cuda()
        if dev.index not in self._ds:
            self._ds[dev.index] = SparseDataset(self.Rc, self.train, dev)
        return self._ds[dev.index]

    def release(self):
        self._ds.clear()

    def construct(self, classifier, *args, **kwargs):
        """classifier(R, M, *args, **kwargs) on these entries."""
        from .bnmf import _TwoFactorBase
        from .bnmtf import _ThreeFactorBase
        from .np_models import _NPBase
        if isinstance(classifier, type) and issubclass(classifier, _NPBase):
            return classifier.from_dataset(self.dataset(), *args, **kwargs)
        if isinstance(classifier, type) and issubclass(classifier, (_TwoFactorBase, _ThreeFactorBase)):
            model = classifier.from_dataset(self.dataset(), *args, seed=0, **kwargs)
            model._seed_after_initialise = True          # see _seeded
            return model
        return classifier(self.Rc, self.mask(), *args, **kwargs)


def _seeded(model):
    """from_dataset() fixes a model's Philox seed when it is called, while a model built by its constructor derives the
    seed from numpy's state when initialise() first reaches the device, after its host draws.  For a model from
    _Entries.construct, derive it now, after initialise(): a seeded Gibbs fit then draws what it draws on dense input."""
    if model.__dict__.pop('_seed_after_initialise', False):
        from . import _lib
        model._seed = model._eng.seed = _lib.derive_seed()
    return model


def _sparse_entries(R, M, validate):
    """The training set of (R, M) as an _Entries (M may be one already: a fold handed down by a cross-validation driver),
    or None for dense input.  validate: the model classes' checks (data.validate_sparse), which dense input meets in the
    constructor of every fit."""
    import scipy.sparse as sp
    from . import data
    if isinstance(M, _Entries):
        return M
    if not sp.issparse(R):
        if sp.issparse(M):
            raise ValueError("with dense R, M must be a dense array, not %s" % type(M).__name__)
        return None
    if validate:
        Rc, _, train = data.validate_sparse(R, M)
        return _Entries(Rc, train)
    if M is not None and not sp.issparse(M):
        raise ValueError("with sparse R, M must be None or a scipy.sparse matrix, not %s" % type(M).__name__)
    Rc = data.canonical_csr(R)
    return _Entries(Rc, mask._selection(Rc, M))


def _as_entries(entries, train):
    """A training set given to a run_model() method: a dense mask as it is, a sparse one as an _Entries."""
    if entries is None or isinstance(train, _Entries):
        return train
    return _Entries(entries.Rc, mask._selection(entries.Rc, train))


def _cv_folds(entries, I, J, no_folds, M):
    """[(training set, test mask)] of the cross-validation drivers: the reference's compute_folds_attempts and
    compute_Ms for dense input; for sparse input an _Entries per fold and a CSR test mask, the same folds."""
    if entries is None:
        folds_test = mask.compute_folds_attempts(I=I, J=J, no_folds=no_folds, attempts=attempts_generate_M, M=M)
        return list(zip(mask.compute_Ms(folds_test), folds_test))
    tests = mask._fold_selections_attempts(entries.Rc, no_folds, attempts_generate_M, entries.train)
    return [(_Entries(entries.Rc, entries.train & ~t), mask._entry_mask(entries.Rc, t)) for t in tests]


class _Search:
    """Shared machinery of the three searches: fit `restarts` models per point, keep the one with the highest
    log-likelihood, record every metric of that one.  Sparse R: every fit shares one resident dataset of M's entries."""

    def __init__(self, classifier, R, M, priors, iterations, restarts, devices):
        self.entries = _sparse_entries(R, M, validate=True)
        self._own_entries = not isinstance(M, _Entries)
        if self.entries is not None:
            R = self.entries.Rc
        self.classifier, self.R, self.M, self.priors = classifier, R, M, priors
        (self.I, self.J) = self.R.shape
        self.iterations, self.restarts = iterations, restarts
        assert self.restarts > 0, "Need at least 1 restart."
        self.pool = DevicePool(devices)

    def _new(self, *args):
        if self.entries is None:
            return self.classifier(self.R, self.M, *args)
        return self.entries.construct(self.classifier, *args)

    def _done(self):
        if self.entries is not None and self._own_entries:
            self.entries.release()

    def _build(self, point):       # -> model, constructed and initialised
        raise NotImplementedError

    def _evaluate(self, points, burn_in, thinning, minimum_TN):
        """{metric: value} of the best restart, for each point, in order."""
        qa = _quality_args(burn_in, thinning)

        def run(model):
            if minimum_TN is None:
                model.run(iterations=self.iterations)
            else:
                model.run(iterations=self.iterations, minimum_TN=minimum_TN)
            return model.quality('loglikelihood', *qa)

        out = []
        if len(self.pool.devices) <= 1:
            for p in points:                                   # the reference's order: build, run, compare
                best, best_ll = None, None
                for _ in range(self.restarts):
                    model = self._build(p)
                    ll = run(model)
                    if best is None or ll > best_ll:
                        best, best_ll = model, ll
                out.append({m: best.quality(m, *qa) for m in metrics})
            return out
        # Several devices: the fits of a WAVE (about one model per device) are built in the reference's order -- so the
        # host random streams keep their positions -- run concurrently, summarised, and their engines released before the
        # next wave is built: only one wave's copies of R / masks / digit planes are resident at a time.
        per_wave = max(1, len(self.pool.devices) // self.restarts)
        for w0 in range(0, len(points), per_wave):
            wave = points[w0:w0 + per_wave]
            models = []
            for p in wave:
                for _ in range(self.restarts):
                    with self.pool.on(len(models)):      # an engine created by initialise() lands on the device map() will use
                        model = self._build(p)
                    _pin_seed(model)
                    models.append(model)
            lls = self.pool.map(run, models)
            for ip in range(len(wave)):
                best, best_ll = None, None
                for r in range(self.restarts):
                    model, ll = models[ip * self.restarts + r], lls[ip * self.restarts + r]
                    if best is None or ll > best_ll:
                        best, best_ll = model, ll
                with _home(best):
                    out.append({m: best.quality(m, *qa) for m in metrics})
            for model in models:                                  # device buffers of this wave (host state stays)
                if hasattr(model, '_eng'):
                    model._eng = None
                model.__dict__.pop('_samples', None)
        return out

    def all_values(self, metric):
        assert metric in metrics, "Unrecognised metric name: %s." % metric
        return self.all_performances[metric]


class LineSearch(_Search):
    """Line search over K for the two-factor models (reference line_search_bnmf.py:38-88)."""

    def __init__(self, classifier, values_K, R, M, priors, initUV, iterations, restarts=1, devices=None):
        _Search.__init__(self, classifier, R, M, priors, iterations, restarts, devices)
        self.values_K, self.initUV = values_K, initUV
        self.all_performances = {metric: [] for metric in metrics}

    def _build(self, K):
        model = self._new(K, self.priors)
        model.initialise(init=self.initUV)
        return _seeded(model)

    def search(self, burn_in=None, thinning=None, minimum_TN=None):
        for res in self._evaluate(self.values_K, burn_in, thinning, minimum_TN):
            for metric in metrics:
                self.all_performances[metric].append(res[metric])
        self._done()

    def best_value(self, metric):
        values = self.all_values(metric)
        return self.values_K[values.index(min(values))]


class GridSearch(_Search):
    """Full (K, L) grid for the tri-factorisation models (reference grid_search_bnmtf.py:43-107).  The scalar
    lambdaF / lambdaS / lambdaG priors are expanded to matrices per grid point, as there."""

    def __init__(self, classifier, values_K, values_L, R, M, priors, initS, initFG, iterations, restarts=1, devices=None):
        _Search.__init__(self, classifier, R, M, priors, iterations, restarts, devices)
        self.values_K, self.values_L, self.initS, self.initFG = values_K, values_L, initS, initFG
        self.all_performances = {metric: np.empty((len(values_K), len(values_L))) for metric in metrics}

    def _build(self, KL):
        K, L = KL
        priors = self.priors.copy()
        priors['lambdaF'] = self.priors['lambdaF'] * np.ones((self.I, K))
        priors['lambdaS'] = self.priors['lambdaS'] * np.ones((K, L))
        priors['lambdaG'] = self.priors['lambdaG'] * np.ones((self.J, L))
        model = self._new(K, L, priors)
        model.initialise(init_S=self.initS, init_FG=self.initFG)
        return _seeded(model)

    def search(self, burn_in=None, thinning=None):
        points = [(K, L) for K in self.values_K for L in self.values_L]
        results = self._evaluate(points, burn_in, thinning, None)
        for idx, res in enumerate(results):
            ik, il = divmod(idx, len(self.values_L))
            for metric in metrics:
                self.all_performances[metric][ik, il] = res[metric]
        self._done()

    def best_value(self, metric):
        index = int(np.argmin(self.all_values(metric)))
        ik, il = divmod(index, len(self.values_L))       # (python-2 integer division in the reference, :105-107)
        return (self.values_K[ik], self.values_L[il])


class GreedySearch(_Search):
    """Greedy walk over the (K, L) grid from its first corner: at each step try K+, L+ and both, move to the best of
    the three unless the current point beats them all; along an edge continue in the remaining direction
    (reference greedy_search_bnmtf.py:47-183).  Every tried point is stored as (K, L, value); the three candidates of
    a step are independent fits and go to the device pool together."""

    def __init__(self, classifier, values_K, values_L, R, M, priors, initS, initFG, iterations, restarts=1, devices=None):
        _Search.__init__(self, classifier, R, M, priors, iterations, restarts, devices)
        self.values_K, self.values_L, self.initS, self.initFG = values_K, values_L, initS, initFG
        self.all_performances = {metric: [] for metric in metrics}

    def _build(self, KL):
        model = self._new(KL[0], KL[1], self.priors)
        model.initialise(init_S=self.initS, init_FG=self.initFG)
        return _seeded(model)

    def find_KL(self, metric, K, L):
        return [x for x in self.all_values(metric) if (x[0], x[1]) == (K, L)]

    def search(self, search_metric, burn_in=None, thinning=None, minimum_TN=None):
        assert search_metric in metrics, "Unrecognised metric name: %s." % search_metric

        def try_points(points):
            new = []
            for p in points:
                if not self.find_KL(search_metric, *p) and p not in new:
                    new.append(p)
            for p, res in zip(new, self._evaluate(new, burn_in, thinning, minimum_TN)):
                for metric in metrics:
                    self.all_performances[metric].append((p[0], p[1], res[metric]))
            return [self.find_KL(search_metric, *p)[0][2] for p in points]

        vK, vL = self.values_K, self.values_L
        ik, il = 0, 0
        p_L = None
        so_far = try_points([(vK[0], vL[0])])[0]
        while ik < len(vK) - 1 and il < len(vL) - 1:
            new_K, new_L = vK[ik + 1], vL[il + 1]
            p_K, p_L, p_KL = try_points([(new_K, vL[il]), (vK[ik], new_L), (new_K, new_L)])
            if so_far < min(p_K, p_L, p_KL):
                break
            if p_K < p_L and p_K < p_KL:
                ik, so_far = ik + 1, p_K
            elif p_L < p_KL:
                il, so_far = il + 1, p_L
            else:
                ik, il, so_far = ik + 1, il + 1, p_KL
        if ik == len(vK) - 1:
            while il < len(vL) - 1:
                p_L = try_points([(vK[ik], vL[il + 1])])[0]
                if so_far < p_L:
                    break
                il, so_far = il + 1, p_L
        elif il == len(vL) - 1:
            while ik < len(vK) - 1:
                p_K = try_points([(vK[ik + 1], vL[il])])[0]
                if so_far < p_K:
                    break
                ik += 1
                # the reference assigns performance_new_L here (greedy_search_bnmtf.py:165): the running best becomes the
                # LAST L-direction score of the main loop, not the score just accepted.  Kept, so that the walk visits
                # the same points; where the reference would hit an unbound name (main loop never ran) use p_K.
                so_far = p_K if p_L is None else p_L
        self._done()

    def best_value(self, metric):
        (best_K, best_L, _) = min(self.all_values(metric), key=lambda x: x[2])
        return (best_K, best_L)


# ---------------------------------------------------------------------------------------------------------------
class _SearchCrossValidation:
    """Folds -> model selection on the training mask -> `restarts` final fits, the one with the best log-likelihood
    predicts the test fold (reference line_search_cross_validation.py:33-135, greedy_search_cross_validation.py:33-142)."""

    def __init__(self, classifier, R, M, folds, priors, iterations, restarts, quality_metric, file_performance, devices):
        self.classifier = classifier
        self.entries = _sparse_entries(R, M, validate=False)
        if self.entries is None:
            self.R = np.array(R, dtype=float)
            self.M = np.array(M)
        else:
            self.R, self.M = self.entries.Rc, M
        self.folds, self.priors, self.iterations, self.restarts = folds, priors, iterations, restarts
        self.quality_metric = quality_metric
        self.fout = open(file_performance, 'w')
        (self.I, self.J) = self.R.shape
        if self.entries is None:
            assert (self.R.shape == self.M.shape), "R and M are of different shapes: %s and %s respectively." % (self.R.shape, self.M.shape)
        assert self.quality_metric in metrics
        self.performances = {}
        self.devices = devices
        self.pool = DevicePool(devices)

    # hooks
    def _select(self, train, burn_in, thinning, minimum_TN):     # -> (all values of the metric, best point)
        raise NotImplementedError

    def _final_model(self, train, point):                         # -> constructed + initialised model
        raise NotImplementedError

    _best_label = "K"

    def run(self, burn_in=None, thinning=None, minimum_TN=None):
        performances_test = {measure: [] for measure in measures}
        for i, (train, test) in enumerate(_cv_folds(self.entries, self.I, self.J, self.folds, self.M)):
            all_performances, best = self._select(train, burn_in, thinning, minimum_TN)
            self.fout.write("All model fits for fold %s, metric %s: %s.\n" % (i + 1, self.quality_metric, all_performances))
            self.fout.flush()
            self.fout.write("Best %s for fold %s: %s.\n" % (self._best_label, i + 1, best))
            performance = self._run_final(train, test, best, burn_in, thinning, minimum_TN)
            self.fout.write("Performance: %s.\n\n" % performance)
            self.fout.flush()
            for measure in measures:
                performances_test[measure].append(performance[measure])
            if self.entries is not None:
                train.release()
        if self.entries is not None:
            self.entries.release()
        self.average_performance_test = self.compute_average_performance(performances_test)
        self.performances = performances_test
        self.fout.write("Average performance: %s. \nPerformances test: %s." % (self.average_performance_test, performances_test))
        self.fout.flush()

    def compute_average_performance(self, performances):
        return {measure: (sum(values) / float(len(values))) for measure, values in performances.items()}

    def _run_final(self, train, test, point, burn_in, thinning, minimum_TN):
        qa = _quality_args(burn_in, thinning)
        train = _as_entries(self.entries, train)

        def fit(model):
            if minimum_TN is None:
                model.run(self.iterations)
            else:
                model.run(self.iterations, minimum_TN=minimum_TN)
            return model.quality('loglikelihood', *qa), model.predict(test, *qa)

        if len(self.pool.devices) <= 1:
            fits = [fit(self._final_model(train, point)) for _ in range(self.restarts)]
        else:
            models = []
            for r in range(self.restarts):
                with self.pool.on(r):
                    models.append(self._final_model(train, point))
                _pin_seed(models[-1])
            fits = self.pool.map(fit, models)
        best_ll, best_perf = None, None
        for ll, perf in fits:
            if best_ll is None or ll > best_ll:
                best_ll, best_perf = ll, perf
        return best_perf


class LineSearchCrossValidation(_SearchCrossValidation):
    def __init__(self, classifier, R, M, values_K, folds, priors, init_UV, iterations, restarts, quality_metric,
                 file_performance, devices=None):
        _SearchCrossValidation.__init__(self, classifier, R, M, folds, priors, iterations, restarts, quality_metric,
                                        file_performance, devices)
        self.values_K, self.init_UV = values_K, init_UV

    def _select(self, train, burn_in, thinning, minimum_TN):
        ls = LineSearch(classifier=self.classifier, values_K=self.values_K, R=self.R, M=train, priors=self.priors,
                        initUV=self.init_UV, iterations=self.iterations, restarts=self.restarts, devices=self.devices)
        ls.search(burn_in=burn_in, thinning=thinning, minimum_TN=minimum_TN)
        return ls.all_values(metric=self.quality_metric), ls.best_value(metric=self.quality_metric)

    def _final_model(self, train, K):
        if isinstance(train, _Entries):
            model = train.construct(self.classifier, K=K, priors=self.priors)
        else:
            model = self.classifier(R=self.R, M=train, K=K, priors=self.priors)
        model.initialise(self.init_UV)
        return _seeded(model)

    def run_model(self, train, test, K, burn_in=None, thinning=None, minimum_TN=None):
        return self._run_final(train, test, K, burn_in, thinning, minimum_TN)


class GreedySearchCrossValidation(_SearchCrossValidation):
    _best_label = "K,L"

    def __init__(self, classifier, R, M, values_K, values_L, folds, priors, init_S, init_FG, iterations, restarts,
                 quality_metric, file_performance, devices=None):
        _SearchCrossValidation.__init__(self, classifier, R, M, folds, priors, iterations, restarts, quality_metric,
                                        file_performance, devices)
        self.values_K, self.values_L, self.init_S, self.init_FG = values_K, values_L, init_S, init_FG

    def _select(self, train, burn_in, thinning, minimum_TN):
        # the reference passes M=self.M (the full mask), not the training fold (greedy_search_cross_validation.py:72): kept
        gs = GreedySearch(classifier=self.classifier, values_K=self.values_K, values_L=self.values_L, R=self.R,
                          M=self.M if self.entries is None else self.entries,
                          priors=self.priors, initS=self.init_S, initFG=self.init_FG, iterations=self.iterations,
                          restarts=self.restarts, devices=self.devices)
        gs.search(self.quality_metric, burn_in=burn_in, thinning=thinning, minimum_TN=minimum_TN)
        return gs.all_values(metric=self.quality_metric), gs.best_value(metric=self.quality_metric)

    def _final_model(self, train, KL):
        if isinstance(train, _Entries):
            model = train.construct(self.classifier, K=KL[0], L=KL[1], priors=self.priors)
        else:
            model = self.classifier(R=self.R, M=train, K=KL[0], L=KL[1], priors=self.priors)
        model.initialise(self.init_S, self.init_FG)
        return _seeded(model)

    def run_model(self, train, test, K, L, burn_in=None, thinning=None, minimum_TN=None):
        return self._run_final(train, test, (K, L), burn_in, thinning, minimum_TN)


# ---------------------------------------------------------------------------------------------------------------
def _fit_fold(job):
    method, X, train, test, parameters, train_config = job
    if isinstance(train, _Entries):          # sparse input: the fold's own dataset, released when its fit is done
        try:
            model = _seeded(train.construct(method, **parameters))     # (counts the seed as dense input does)
            model.train(**train_config)
            return model.predict(test)
        finally:
            train.release()
    model = method(X, train, **parameters)
    model.train(**train_config)
    return model.predict(test)


class MatrixCrossValidation:
    """K-fold cross-validation of `method(X, train, **parameters).train(**train_config).predict(test)` over a list of
    parameter dicts (reference matrix_cross_validation.py:44-148).  The folds of one parameter setting are independent
    fits and are spread over the devices of `devices` (default: one, i.e. the reference's sequential order)."""

    def __init__(self, method, X, M, K, parameter_search, train_config, file_performance, devices=1):
        self.method = method
        self.entries = _sparse_entries(X, M, validate=False)
        if self.entries is None:
            self.X = np.array(X, dtype=float)
            self.M = np.array(M)
        else:
            self.X, self.M = self.entries.Rc, M
        self.K, self.train_config, self.parameter_search = K, train_config, parameter_search
        self.fout = open(file_performance, 'w')
        (self.I, self.J) = self.X.shape
        if self.entries is None:
            assert (self.X.shape == self.M.shape), "X and M are of different shapes: %s and %s respectively." % (self.X.shape, self.M.shape)
        self.all_performances = {}        # JSON(parameters) -> {criterion: [per fold]}
        self.average_performances = {}    # JSON(parameters) -> {criterion: average}
        self.performances = {}            # criterion -> [average per parameter setting]
        self.pool = DevicePool(devices)

    def run(self):
        for parameters in self.parameter_search:
            try:
                folds = _cv_folds(self.entries, self.I, self.J, self.K, self.M)
                self.all_performances[self.JSON(parameters)] = {}
                jobs = [(self.method, self.X, train, test, parameters, self.train_config) for train, test in folds]
                for performance_dict in self.pool.map(_fit_fold, jobs):
                    self.store_performances(performance_dict, parameters)
                self.log(parameters)
            except Exception as e:
                self.fout.write("Tried parameters %s but got exception: %s. \n" % (parameters, e))
                self.fout.flush()

    def run_model(self, train, test, parameters):
        return _fit_fold((self.method, self.X, _as_entries(self.entries, train), test, parameters, self.train_config))

    def JSON(self, d):
        return json.dumps({k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in d.items()}, sort_keys=True)

    def store_performances(self, performance_dict, parameters):
        store = self.all_performances[self.JSON(parameters)]
        for name, value in performance_dict.items():
            store.setdefault(name, []).append(value)

    def compute_average_performances(self, parameters):
        performances = self.all_performances[self.JSON(parameters)]
        average = {name: (sum(values) / float(len(values))) for name, values in performances.items()}
        self.average_performances[self.JSON(parameters)] = average
        for name, value in average.items():
            self.performances.setdefault(name, []).append(value)

    def find_best_parameters(self, evaluation_criterion, low_better):
        pick = min if low_better else max
        self.best_performance = pick(self.performances[evaluation_criterion])
        index_best = self.performances[evaluation_criterion].index(self.best_performance)
        self.best_parameters = self.parameter_search[index_best]
        self.best_performances_all = self.average_performances[self.JSON(self.best_parameters)]
        self.log_best(index_best)
        return (self.best_parameters, self.best_performance)

    def log(self, parameters):
        self.compute_average_performances(parameters)
        key = self.JSON(parameters)
        self.fout.write("Tried parameters %s. Average performances: %s. \nAll performances: %s. \n" %
                        (parameters, self.average_performances[key], self.all_performances[key]))
        self.fout.flush()

    def log_best(self, index_best):
        self.fout.write("Best performances: %s. Best parameters: %s. \n" % (self.best_performances_all, self.best_parameters))
        self.fout.flush()


class ParallelMatrixCrossValidation(MatrixCrossValidation):
    """Reference parallel_matrix_cross_validation.py:44-76 runs the folds in a multiprocessing.Pool(P); here P is the
    number of GPUs to spread them over (capped by the GPUs present)."""

    def __init__(self, method, X, M, K, parameter_search, train_config, file_performance, P):
        MatrixCrossValidation.__init__(self, method, X, M, K, parameter_search, train_config, file_performance, devices=P)
        self.P = P


class MatrixNestedCrossValidation:
    """Outer K folds; on each training mask an inner ParallelMatrixCrossValidation picks the parameters with the
    lowest average MSE (first setting if nothing could be evaluated), one model is fit with them and scored on the
    outer test fold (reference nested_matrix_cross_validation.py:51-133)."""

    def __init__(self, method, X, M, K, P, parameter_search, train_config, file_performance, files_nested_performances):
        self.method = method
        self.entries = _sparse_entries(X, M, validate=False)
        if self.entries is None:
            self.X = np.array(X, dtype=float)
            self.M = np.array(M)
        else:
            self.X, self.M = self.entries.Rc, M
        self.K, self.P, self.train_config, self.parameter_search = K, P, train_config, parameter_search
        self.files_nested_performances = files_nested_performances
        self.fout = open(file_performance, 'w')
        (self.I, self.J) = self.X.shape
        if self.entries is None:
            assert (self.X.shape == self.M.shape), "X and M are of different shapes: %s and %s respectively." % (self.X.shape, self.M.shape)
        self.all_performances = {}
        self.average_performances = {}

    def run(self):
        for i, (train, test) in enumerate(_cv_folds(self.entries, self.I, self.J, self.K, self.M)):
            crossval = ParallelMatrixCrossValidation(method=self.method, X=self.X, M=train, K=self.K,
                                                     parameter_search=self.parameter_search, train_config=self.train_config,
                                                     file_performance=self.files_nested_performances[i], P=self.P)
            crossval.run()
            try:
                (best_parameters, _) = crossval.find_best_parameters(evaluation_criterion='MSE', low_better=True)
            except KeyError:
                best_parameters = self.parameter_search[0]
            performance_dict = self.run_model(train, test, best_parameters)
            self.store_performances(performance_dict)
        self.log()

    def run_model(self, train, test, parameters):
        return _fit_fold((self.method, self.X, _as_entries(self.entries, train), test, parameters, self.train_config))

    def store_performances(self, performance_dict):
        for name, value in performance_dict.items():
            self.all_performances.setdefault(name, []).append(value)

    def compute_average_performances(self):
        self.average_performances = {name: (sum(values) / float(len(values))) for name, values in self.all_performances.items()}

    def log(self):
        self.compute_average_performances()
        self.fout.write("Average performances: %s. \nAll performances: %s. \n" % (self.average_performances, self.all_performances))
        self.fout.flush()
