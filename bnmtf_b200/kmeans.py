"""K-means with missing values, used for init_FG='kmeans' (host-side port of the behaviour of
code/models/kmeans/kmeans.py:6-205; one-off initialisation, outside the update sweep -- SURVEY.md section 8f #2).

Semantics kept: centroids drawn with python's `random.uniform` between the per-coordinate min and max of the
observed values (same call order, so a seeded run picks the same centroids); distance = mean squared difference
over the coordinates observed in both the point and the centroid (None / infinite when there is no overlap, ties go
to the lowest cluster index); centroid = per-coordinate mean of the observed values of its points (coordinate masked
out when none is observed); an empty cluster takes the point currently furthest from its centroid ('singleton');
stop when no assignment changes or after 200 iterations; result = one-hot assignment matrix.

One reference quirk is kept on purpose, because it changes the clustering in about a third of seeded runs on the toy
data: the 'singleton' rule binds the empty cluster's centroid to the ROW OF X ITSELF (kmeans.py:149,
`self.centroids[c] = self.X[index_furthest_away]`, a numpy view of the model's private copy of X), so every later
centroid update of that cluster (kmeans.py:170) also overwrites that data point.  Here the centroids are a list of row
arrays as well, and the singleton rule stores the view, so the same write-through happens.

The assignment step -- the no_points x K x no_coordinates part, everything else is O(K x no_coordinates) bookkeeping -- runs
on the GPU when a device is given (csrc/kmeans.cu through bnmtf_kmeans_distances_f64: the same bits as the numpy
expression in _all_distances, so the clustering is the same); the model classes always pass their device.  Without a
device the class is the plain host port (tests/test_kmeans.py pins it against the reference's goldens on CPU).
"""
import random

import numpy as np

MAX_ITERATIONS = 200


class KMeans(object):
    def __init__(self, X, M, K, resolve_empty='singleton', device=None):
        self.device = device
        self._dev = None                # (X, M, centroid, mask, distance) device tensors, made on first use
        self._aliased = set()           # rows of X a centroid is a view of (they change under update_cluster)
        self.X = np.array(X, dtype=float)
        self.M = np.array(M, dtype=float)
        self.K = K
        self.resolve_empty = resolve_empty
        assert len(self.X.shape) == 2, "Input matrix X is not a two-dimensional array, but instead %s-dimensional." % len(self.X.shape)
        assert self.X.shape == self.M.shape, "Input matrix X is not of the same size as the indicator matrix M: %s and %s respectively." % (self.X.shape, self.M.shape)
        assert self.K > 0, "K should be greater than 0."
        (self.no_points, self.no_coordinates) = self.X.shape
        self.no_unique_points = len(set(tuple(row) for row in self.X.tolist()))
        for i, c in enumerate(self.M.sum(axis=1)):
            assert c != 0, "Fully unobserved row in X, row %s." % i
        keep = self.M.sum(axis=0) != 0
        if not keep.all():
            self.X, self.M = self.X[:, keep], self.M[:, keep]
            self.no_coordinates = self.X.shape[1]
        self.distances = np.zeros(self.no_points)

    def initialise(self, seed=None):
        if seed is not None:
            random.seed(seed)
        obs = self.M != 0
        self.mins = [self.X[obs[:, j], j].min() for j in range(self.no_coordinates)]
        self.maxs = [self.X[obs[:, j], j].max() for j in range(self.no_coordinates)]
        self.centroids = [np.array(self.random_cluster_centroid(), dtype=float) for _ in range(self.K)]
        self.cluster_assignments = np.full(self.no_points, -1, dtype=int)
        self.mask_centroids = np.ones((self.K, self.no_coordinates))

    def random_cluster_centroid(self):
        return [random.uniform(self.mins[c], self.maxs[c]) for c in range(self.no_coordinates)]

    def cluster(self):
        iteration = 1
        change = True
        while change:
            iteration += 1
            change = self.assignment()
            self.update()
            if iteration >= MAX_ITERATIONS:
                break
        self.create_matrix()

    def _all_distances_device(self):
        import torch
        from . import _lib
        from .engine import _ptr, _stream
        n, d, K = self.no_points, self.no_coordinates, self.K
        if self._dev is None:
            dev = torch.device(self.device)
            f = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
            self._dev = {"X": f(self.X), "M": f(self.M), "C": torch.empty((K, d), dtype=torch.float64, device=dev),
                         "MC": torch.empty((K, d), dtype=torch.float64, device=dev),
                         "D": torch.empty((n, K), dtype=torch.float64, device=dev)}
        t = self._dev
        for i in sorted(self._aliased):                 # data points overwritten through a centroid view (see top)
            t["X"][i].copy_(torch.from_numpy(np.ascontiguousarray(self.X[i])))
        t["C"].copy_(torch.from_numpy(np.stack(self.centroids)))
        t["MC"].copy_(torch.from_numpy(np.ascontiguousarray(self.mask_centroids, dtype=np.float64)))
        with torch.cuda.device(t["X"].device):
            _lib.call("bnmtf_kmeans_distances_f64", _ptr(t["X"]), _ptr(t["M"]), n, d, _ptr(t["C"]), _ptr(t["MC"]), K, _ptr(t["D"]),
                      _stream())
        return t["D"].cpu().numpy()

    def _all_distances(self):
        """no_points x K matrix of masked mean squared differences (inf where nothing overlaps)."""
        if self.device is not None:
            return self._all_distances_device()
        both = self.M[:, None, :] * self.mask_centroids[None, :, :]
        overlap = both.sum(axis=2)
        sq = (both * (self.X[:, None, :] - np.stack(self.centroids)[None, :, :]) ** 2).sum(axis=2)
        with np.errstate(all='ignore'):
            return np.where(overlap > 0, sq / overlap, np.inf)

    def assignment(self):
        dist = self._all_distances()
        new = dist.argmin(axis=1)                       # first minimum = lowest index on ties
        best = dist[np.arange(self.no_points), new]
        self.distances = np.where(np.isfinite(best), best, 0.0)
        change = bool((new != self.cluster_assignments).any())
        self.cluster_assignments = new
        self.data_point_assignments = [list(np.nonzero(new == c)[0]) for c in range(self.K)]
        return change

    def update(self):
        for c in range(self.K):
            self.update_cluster(c)

    def update_cluster(self, c):
        members = self.data_point_assignments[c]
        if len(members) == 0:
            if self.no_unique_points >= self.K:
                if self.resolve_empty == 'singleton':
                    far = int(self.distances.argmax())
                    old = int(self.cluster_assignments[far])
                    self.centroids[c] = self.X[far]          # a VIEW: later updates of c write through into X (see top)
                    self._aliased.add(far)
                    self.mask_centroids[c] = self.M[far]
                    self.distances[far] = 0.0
                    self.cluster_assignments[far] = c
                    self.data_point_assignments[c] = [far]
                    self.data_point_assignments[old].remove(far)
                    self.update_cluster(old)
                else:
                    self.centroids[c] = np.array(self.random_cluster_centroid(), dtype=float)
                    self.mask_centroids[c] = np.ones(self.no_coordinates)
            return
        Xc, Mc = self.X[members], self.M[members]
        counts = Mc.sum(axis=0)
        with np.errstate(all='ignore'):
            means = np.where(counts > 0, (Mc * Xc).sum(axis=0) / counts, 0.0)
        self.centroids[c][:] = means                         # in place, like the reference's per-coordinate writes
        self.mask_centroids[c] = (counts > 0).astype(float)

    def create_matrix(self):
        self.clustering_results = np.zeros((self.no_points, self.K))
        self.clustering_results[np.arange(self.no_points), self.cluster_assignments] = 1


# ==== K-means on the observed entries of a scipy.sparse matrix ===================================================
def _splitmix(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def unique_dense_rows(A):
    """len(set(tuple(row) for row in A.toarray())) of a canonical scipy CSR A without the dense array: zero entries are
    dropped (they equal absent ones), every row is keyed by its entry count and two order-free 64-bit hashes of its
    (column, value bits) pairs, and rows with equal keys are compared entry by entry; only a hash collision (never seen)
    takes the exact per-row path."""
    n = A.shape[0]
    nz = A.data != 0
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(A.indptr))[nz]
    cols = A.indices[nz].astype(np.uint64)
    bits = np.ascontiguousarray(A.data[nz], dtype=np.float64).view(np.uint64)
    cnt = np.bincount(rows, minlength=n)
    ptr = np.concatenate([[0], np.cumsum(cnt)])
    keys = [cnt.astype(np.uint64)]
    for salt in (np.uint64(0x632BE59BD9B4E019), np.uint64(0x8CB92BA72F3D8DD7)):
        h = _splitmix(_splitmix(cols ^ salt) ^ bits)
        cs = np.concatenate([[np.uint64(0)], np.cumsum(h, dtype=np.uint64)])
        keys.append(cs[ptr[1:]] - cs[ptr[:-1]])
    keys = np.stack(keys, axis=1)
    order = np.lexsort(keys.T[::-1])
    ks = keys[order]
    same = (ks[1:] == ks[:-1]).all(axis=1)
    a, b = order[:-1][same], order[1:][same]             # neighbours with equal keys: must be equal rows
    if a.size:
        la = cnt[a]
        ea = np.repeat(ptr[a], la) + (np.arange(int(la.sum())) - np.repeat(np.cumsum(la) - la, la))
        eb = ea - np.repeat(ptr[a], la) + np.repeat(ptr[b], la)
        if not (np.array_equal(cols[ea], cols[eb]) and np.array_equal(bits[ea], bits[eb])):
            return len(set(tuple(row) for row in (A[i].toarray()[0].tolist() for i in range(n))))
    return int(n - same.sum())


class SparseKMeans(KMeans):
    """KMeans on the observed entries of a sparse matrix: the clusterings, centroids and masks of KMeans on the dense pair
    (X_all.toarray(), 0/1 pattern of X), with nothing of size no_points x no_coordinates on the host or the device.

    X: scipy.sparse CSR (canonical: sorted, duplicate-free) of the observed entries -- every stored entry is observed,
    explicit zeros included.  X_all: the matrix whose dense rows are the data points (default X; with a training mask it is
    all of R, the test entries included): it decides no_unique_points and the values a 'singleton' centroid starts from.

    The device does the two O(nnz) steps: bnmtf_csr_kmeans_distances_f64 (the dense kernel's bits) over the points' CSR, and
    bnmtf_csr_kmeans_sums_f64 (numpy's member-order axis-0 sums) over the coordinate-major CSR.  The reference quirk of
    KMeans is kept: a 'singleton' centroid is a view of the dense row of its point (materialised on the host for that point
    only), later updates of the centroid write through into that point's data, and the point's values in both device value
    arrays (K-means' own copies) follow.  A cluster summed after such a write and containing the point, or whose membership
    the singleton rule changed, is summed again on its own, so the sequence of KMeans.update is reproduced exactly."""

    def __init__(self, X, K, X_all=None, resolve_empty='singleton', device=None):
        import scipy.sparse as sp
        from .data import canonical_csr
        if device is None:
            raise ValueError("SparseKMeans runs on a CUDA device: give `device`")
        self.device = device
        self.K = K
        self.resolve_empty = resolve_empty
        assert self.K > 0, "K should be greater than 0."
        X = canonical_csr(X)
        X_all = X if X_all is None else canonical_csr(X_all)
        if tuple(X_all.shape) != tuple(X.shape):
            raise ValueError("X_all has shape %s, X has %s" % (tuple(X_all.shape), tuple(X.shape)))
        (self.no_points, d_all) = X.shape
        self.no_unique_points = unique_dense_rows(X_all)
        per_row = np.diff(X.indptr)
        if (per_row == 0).any():
            assert False, "Fully unobserved row in X, row %s." % int(np.argmin(per_row != 0))
        keep = np.bincount(X.indices, minlength=d_all) != 0
        self._keep = keep
        newcol = (np.cumsum(keep) - 1).astype(np.int32)
        self.no_coordinates = d = int(keep.sum())
        self._Xall = X_all
        # the points' CSR (row i = point i over the kept coordinates) and the coordinate-major CSR; perm[e]: position of
        # point-major entry e in the coordinate-major arrays
        self._ptr = np.asarray(X.indptr, dtype=np.int64)
        self._col = newcol[X.indices]
        self._val = np.array(X.data, dtype=np.float64)
        P = sp.csr_matrix((np.arange(X.nnz, dtype=np.float64), self._col, self._ptr), shape=(self.no_points, d)).tocsc()
        self._cptr = np.asarray(P.indptr, dtype=np.int64)
        self._pt = np.asarray(P.indices, dtype=np.int32)
        self._inv = P.data.astype(np.int64)             # coordinate-major entry -> point-major entry
        self._perm = np.empty(X.nnz, dtype=np.int64)
        self._perm[self._inv] = np.arange(X.nnz, dtype=np.int64)
        self._rows = {}                 # point -> its dense row (a 'singleton' centroid is a view of it)
        self._alias = {}                # cluster -> the point its centroid is a view of
        self._dirty = set()             # points whose device values lag behind their dense row
        self._dev = None
        if d == 1:                      # every point observes the one coordinate: the data are n x 1
            self._X1 = self._val.reshape(-1, 1).copy()
        self.distances = np.zeros(self.no_points)

    def initialise(self, seed=None):
        if seed is not None:
            random.seed(seed)
        vT = self._val[self._inv]
        self.mins = np.minimum.reduceat(vT, self._cptr[:-1]).tolist()
        self.maxs = np.maximum.reduceat(vT, self._cptr[:-1]).tolist()
        self.centroids = [np.array(self.random_cluster_centroid(), dtype=float) for _ in range(self.K)]
        self.cluster_assignments = np.full(self.no_points, -1, dtype=int)
        self.mask_centroids = np.ones((self.K, self.no_coordinates))

    # ---- device state ----------------------------------------------------------------------------------------
    def _device(self):
        import torch
        if self._dev is None:
            dev = torch.device(self.device)
            t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
            n, d, K = self.no_points, self.no_coordinates, self.K
            f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
            self._dev = {"ptr": t(self._ptr, np.int64), "col": t(self._col, np.int32), "val": t(self._val, np.float64),
                         "cptr": t(self._cptr, np.int64), "pt": t(self._pt, np.int32),
                         "valT": t(self._val[self._inv], np.float64), "C": f64(K, d), "MC": f64(K, d),
                         "D": f64(n, K), "assign": torch.zeros(n, dtype=torch.int32, device=dev),
                         "S": f64(K, d) if d > 1 else None, "N": f64(K, d) if d > 1 else None}
        return self._dev

    def _row(self, p):
        """The dense row of point p (over the kept coordinates), created on first use from X_all."""
        if self.no_coordinates == 1:
            return self._X1[p]
        if p not in self._rows:
            A = self._Xall
            lo, hi = A.indptr[p], A.indptr[p + 1]
            r = np.zeros(self._keep.shape[0])
            r[A.indices[lo:hi]] = A.data[lo:hi]
            self._rows[p] = r[self._keep]
        return self._rows[p]

    def _mask_row(self, p):
        m = np.zeros(self.no_coordinates)
        m[self._col[self._ptr[p]:self._ptr[p + 1]]] = 1.0
        return m

    def _sync_points(self):
        """Device values of the points written through a centroid view <- their dense rows."""
        import torch
        t = self._device()
        for p in sorted(self._dirty):
            lo, hi = int(self._ptr[p]), int(self._ptr[p + 1])
            v = np.ascontiguousarray(self._row(p)[self._col[lo:hi]], dtype=np.float64)
            self._val[lo:hi] = v
            vd = torch.from_numpy(v).to(t["val"].device)
            t["val"][lo:hi].copy_(vd)
            t["valT"].index_copy_(0, torch.from_numpy(self._perm[lo:hi]).to(vd.device), vd)
        self._dirty.clear()

    def _all_distances(self):
        import torch
        from . import _lib
        from .engine import _ptr, _stream
        t = self._device()
        self._sync_points()
        t["C"].copy_(torch.from_numpy(np.stack(self.centroids)))
        t["MC"].copy_(torch.from_numpy(np.ascontiguousarray(self.mask_centroids, dtype=np.float64)))
        with torch.cuda.device(t["D"].device):
            _lib.call("bnmtf_csr_kmeans_distances_f64", _ptr(t["ptr"]), _ptr(t["col"]), _ptr(t["val"]), self.no_points,
                      self.no_coordinates, _ptr(t["C"]), _ptr(t["MC"]), self.K, _ptr(t["D"]), _stream())
        return t["D"].cpu().numpy()

    def _sums(self, only):
        """Device sums / counts of every cluster (only < 0) or of cluster `only`, current data and assignment."""
        import torch
        from . import _lib
        from .engine import _ptr, _stream
        t = self._device()
        self._sync_points()
        t["assign"].copy_(torch.from_numpy(self.cluster_assignments.astype(np.int32)))
        with torch.cuda.device(t["S"].device):
            _lib.call("bnmtf_csr_kmeans_sums_f64", _ptr(t["cptr"]), _ptr(t["pt"]), _ptr(t["valT"]), self.no_coordinates,
                      _ptr(t["assign"]), self.K, int(only), _ptr(t["S"]), _ptr(t["N"]), _stream())
        if only < 0:
            self._S, self._N = t["S"].cpu().numpy(), t["N"].cpu().numpy()
        else:
            self._S[only], self._N[only] = t["S"][only].cpu().numpy(), t["N"][only].cpu().numpy()

    # ---- update step ------------------------------------------------------------------------------------------
    def update(self):
        if self.no_coordinates > 1:
            self._sums(-1)
        self._fresh = set(range(self.K))          # clusters whose sums are those of the current data and membership
        self._changed = set()                     # points written through a centroid since the sums were taken
        for c in range(self.K):
            self.update_cluster(c)

    def update_cluster(self, c):
        members = self.data_point_assignments[c]
        if len(members) == 0:
            if self.no_unique_points >= self.K:
                if self.resolve_empty == 'singleton':
                    far = int(self.distances.argmax())
                    old = int(self.cluster_assignments[far])
                    self.centroids[c] = self._row(far)        # a VIEW of the point's data (see KMeans)
                    self._alias[c] = far
                    self.mask_centroids[c] = self._mask_row(far)
                    self.distances[far] = 0.0
                    self.cluster_assignments[far] = c
                    self.data_point_assignments[c] = [far]
                    self.data_point_assignments[old].remove(far)
                    self._fresh.discard(old)
                    self._fresh.discard(c)
                    self.update_cluster(old)
                else:
                    self.centroids[c] = np.array(self.random_cluster_centroid(), dtype=float)
                    self._alias.pop(c, None)
                    self.mask_centroids[c] = np.ones(self.no_coordinates)
            return
        if self.no_coordinates == 1:                       # numpy sums the contiguous column pairwise: on the host
            Xc = self._X1[members]
            Mc = np.ones_like(Xc)
            counts, sums = Mc.sum(axis=0), (Mc * Xc).sum(axis=0)
        else:
            if c not in self._fresh or any(self.cluster_assignments[p] == c for p in self._changed):
                self._sums(c)
                self._fresh.add(c)
            counts, sums = self._N[c], self._S[c]
        with np.errstate(all='ignore'):
            means = np.where(counts > 0, sums / counts, 0.0)
        self.centroids[c][:] = means                         # in place: writes through into an aliased point
        self.mask_centroids[c] = (counts > 0).astype(float)
        p = self._alias.get(c)
        if p is not None:
            self._dirty.add(p)
            self._changed.add(p)
