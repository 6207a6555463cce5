"""Sparse input of the tri-factor models without a GPU: constructor validation, from_dataset's engine choice, and numpy
restatements of the two K-means kernels of csrc/kmeans.cu (bnmtf_csr_kmeans_distances_f64's walk over the observed leaves of
numpy's pairwise tree, bnmtf_csr_kmeans_sums_f64's member-order sums) against the dense host evaluation they must equal."""
import numpy as np
import pytest
import scipy.sparse as sp

import bnmtf_b200
from bnmtf_b200.kmeans import KMeans, unique_dense_rows

PRI = {"alpha": 1.0, "beta": 1.0, "lambdaF": 1.0, "lambdaS": 1.0, "lambdaG": 1.0}
CLASSES = [bnmtf_b200.bnmtf_gibbs_optimised, bnmtf_b200.bnmtf_vb_optimised, bnmtf_b200.nmtf_icm]


def small():
    R = sp.coo_matrix(([1.0, 0.0, 2.0, 3.0, 4.0], ([0, 0, 1, 2, 2], [0, 2, 1, 0, 2])), shape=(3, 3))
    return R


@pytest.mark.parametrize("cls", CLASSES)
def test_constructor_on_sparse_input(cls):
    R = small()
    m = cls(R, None, 2, 3, PRI)
    assert m._sparse and m.size_Omega == 5.0 and (m.I, m.J) == (3, 3)
    assert m.lambdaF.shape == (3, 2) and m.lambdaS.shape == (2, 3) and m.lambdaG.shape == (3, 3)
    M = sp.csr_matrix(([1.0, 1.0, 1.0, 1.0], ([0, 1, 2, 2], [0, 1, 0, 2])), shape=(3, 3))
    assert cls(sp.csr_array(R), M, 2, 2, PRI).size_Omega == 4.0


@pytest.mark.parametrize("cls", CLASSES)
def test_constructor_messages_on_sparse_input(cls):
    R = small()
    with pytest.raises(AssertionError, match="Fully unobserved row in R, row 1."):
        cls(sp.csr_matrix(([1.0, 2.0], ([0, 2], [0, 1])), shape=(3, 2)), None, 1, 1, PRI)
    with pytest.raises(AssertionError, match="Fully unobserved column in R, column 1."):
        cls(sp.csr_matrix(([1.0, 2.0], ([0, 1], [0, 0])), shape=(2, 2)), None, 1, 1, PRI)
    with pytest.raises(AssertionError, match="not of the same size"):
        cls(R, sp.csr_matrix((2, 3)), 1, 1, PRI)
    with pytest.raises(ValueError, match="more than one stored entry"):
        cls(sp.coo_matrix(([1.0, 2.0, 3.0], ([0, 0, 1], [0, 0, 1])), shape=(2, 2)), None, 1, 1, PRI)
    with pytest.raises(ValueError, match="not a stored entry"):
        cls(R, sp.csr_matrix(([1.0], ([1], [0])), shape=(3, 3)), 1, 1, PRI)
    with pytest.raises(AssertionError, match="Prior matrix lambdaF has the wrong shape"):
        cls(R, None, 2, 2, dict(PRI, lambdaF=np.ones((2, 2))))


def test_dense_constructor_is_unchanged():
    m = bnmtf_b200.bnmtf_vb_optimised(np.ones((2, 3)), np.ones((2, 3)), 1, 1, PRI)
    assert not m._sparse and isinstance(m.R, np.ndarray) and m.size_Omega == 6.0


@pytest.mark.parametrize("cls", CLASSES)
def test_from_dataset_picks_the_sparse_engine(cls, monkeypatch):
    from bnmtf_b200 import bnmtf as tri
    from bnmtf_b200.engine import SparseDataset
    seen = []

    def fake_init(self, dataset, K, L, mode, alpha, beta, seed=0):
        seen.append((type(self).__name__, K, L, mode, alpha, beta, seed))
    monkeypatch.setattr(tri.SparseBNMTFEngine, "__init__", fake_init)
    ds = SparseDataset.__new__(SparseDataset)
    ds.I, ds.J, ds.n_obs, ds.device = 4, 3, 7.0, "cuda:0"
    m = cls.from_dataset(ds, 2, 3, dict(PRI, alpha=2.0), seed=5)
    assert seen == [("SparseBNMTFEngine", 2, 3, cls._mode, 2.0, 1.0, 5)]
    assert m._sparse and m.R is None and m.size_Omega == 7.0 and (m.I, m.J) == (4, 3)
    assert m.lambdaF.shape == (4, 2) and m.lambdaS.shape == (2, 3) and m.lambdaG.shape == (3, 3)


# ---- the sparse distance walk ---------------------------------------------------------------------------------------
def block(terms, pos, lo, n):
    """km_csr_block: the present leaves (positions pos, ascending, in [lo, lo + n)) of one block of <= 128."""
    if n < 8:
        r = 0.0
        for t in terms:
            r = r + t
        return r
    r = [0.0] * 8
    main_end = lo + n - n % 8
    k = 0
    while k < len(pos) and pos[k] < main_end:
        q = (pos[k] - lo) % 8
        r[q] = r[q] + terms[k]
        k += 1
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for t in terms[k:]:
        res = res + t
    return res


def walk(terms, pos, lo, n):
    """km_csr_pairwise: numpy's pairwise tree over positions [lo, lo + n), empty subtrees = +0."""
    if len(pos) == 0:
        return 0.0
    if n <= 128:
        return block(terms, pos, lo, n)
    n2 = n // 2
    n2 -= n2 % 8
    k = int(np.searchsorted(pos, lo + n2))
    return walk(terms[:k], pos[:k], lo, n2) + walk(terms[k:], pos[k:], lo + n2, n - n2)


def sparse_distance(x, m, c, mc):
    """Distance of one point from its observed entries only (m 0/1), as the kernel computes it."""
    pos = np.nonzero(m)[0]
    terms = [float(mc[j] * ((x[j] - c[j]) * (x[j] - c[j]))) for j in pos]
    overlap = float(np.sum(mc[pos]))
    return walk(terms, list(pos), 0, len(x)) / overlap if overlap > 0 else np.inf


def patterns(d, rng):
    yield rng.rand(d) < 0.3
    yield rng.rand(d) < 0.02
    yield np.ones(d, bool)
    m = np.zeros(d, bool)
    m[d - d % 8:] = True                              # leaves only in the tail of the last block
    m[-1] = True
    yield m
    m = rng.rand(d) < 0.5
    m[: d // 2] = False                               # all-empty blocks in front
    m[d // 2] = True
    yield m


@pytest.mark.parametrize("d", [1, 2, 7, 8, 9, 15, 16, 127, 128, 129, 136, 257, 300, 1000, 1029, 4099, 8200, 32768])
def test_sparse_walk_has_the_dense_bits(d):
    rng = np.random.RandomState(d)
    K = 3
    for m in patterns(d, rng):
        if not m.any():
            continue
        X = np.where(m, rng.normal(size=d) * 3.0, 0.0)[None, :]
        M = m.astype(float)[None, :]
        C = rng.normal(size=(K, d))
        MC = (rng.rand(K, d) < 0.8).astype(float)
        MC[2] = 0.0
        MC[2, -1] = 1.0
        km = KMeans(np.ones((1, d)), np.ones((1, d)), K)
        km.X, km.M = X, M                            # zero-filled point, 0/1 mask (columns of M may be empty here)
        km.centroids, km.mask_centroids = list(C), MC
        dense = km._all_distances()[0]
        for c in range(K):
            got = sparse_distance(X[0], M[0], C[c], MC[c])
            assert np.float64(got).tobytes() == np.float64(dense[c]).tobytes(), (d, c, got, dense[c])


# ---- member-order sums -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(3, 2), (50, 5), (1000, 17), (4099, 64), (20000, 3), (300, 622), (40, 2000)])
def test_member_order_sums_are_numpys_axis0_sum(n, d):
    rng = np.random.RandomState(n + d)
    X = rng.normal(size=(n, d)) * np.exp(3 * rng.normal(size=(n, 1)))
    M = (rng.rand(n, d) < 0.4).astype(float)
    X = X * M
    members = np.sort(rng.choice(n, size=max(1, n // 3), replace=False))
    Xc, Mc = X[members], M[members]
    want = (Mc * Xc).sum(axis=0)
    got = np.zeros(d)
    cnt = np.zeros(d)
    for j in range(d):                                 # the kernel: coordinate j, its points in ascending order
        for i in members:
            if M[i, j]:
                got[j] = got[j] + X[i, j]
                cnt[j] += 1.0
    assert np.array_equal(cnt, Mc.sum(axis=0))
    assert np.array_equal(np.where(cnt > 0, got, 0.0), np.where(cnt > 0, want, 0.0))


def test_unique_dense_rows_counts_as_the_dense_set():
    rng = np.random.RandomState(0)
    A = (rng.rand(300, 40) < 0.1) * rng.randint(0, 3, size=(300, 40)).astype(float)
    A[10] = A[20]
    A[30] = 0.0
    A[31] = 0.0
    A[5, 7] = 0.0
    S = sp.csr_matrix(A)
    at = S.indptr[6]
    S = sp.csr_matrix((np.insert(S.data, at, 0.0), np.insert(S.indices, at, 7), np.append(S.indptr[:6], S.indptr[6:] + 1)),
                      shape=S.shape)                   # an explicit zero at (5, 7): equal to an absent entry
    S.sort_indices()
    assert unique_dense_rows(S) == len(set(tuple(r) for r in S.toarray().tolist()))
