"""Sparse input on the host, without a GPU: validation and canonical form of scipy.sparse (R, M), the CSR / CSC build and
the static work plan of the CSR statistics kernel, and a numpy restatement of what that kernel computes (chunk
partials added in chunk order) against the dense masked statistics behind the oracle's conditional parameters."""
import numpy as np
import pytest
import scipy.sparse as sp

PRI = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}


def classes():
    import bnmtf_b200
    return (bnmtf_b200.bnmf_gibbs_optimised, bnmtf_b200.bnmf_vb_optimised, bnmtf_b200.nmf_icm)


def small():
    R = sp.coo_matrix((np.array([1.0, 0.0, 2.0, 3.0, 0.5]), (np.array([0, 0, 1, 2, 2]), np.array([0, 2, 1, 0, 2]))), shape=(3, 3))
    return R


def test_explicit_zeros_are_known_entries():
    for cls in classes():
        m = cls(small(), None, 2, PRI)
        assert m.size_Omega == 5.0
        assert sp.isspmatrix_csr(m.R) and m.R.nnz == 5 and m.M.nnz == 5
        assert m.R[0, 2] == 0.0 and (0, 2) in set(zip(*m.M.nonzero()))
        M = sp.coo_matrix((np.ones(4), ([0, 0, 1, 2], [0, 2, 1, 0])), shape=(3, 3))
        m = cls(small(), M, 2, PRI)
        assert m.size_Omega == 4.0 and m.R.nnz == 5        # R keeps the test entry (2, 2)


@pytest.mark.parametrize("fmt", ["csr", "csc", "coo", "lil", "dok", "bsr", "csr_array"])
def test_any_format_gives_the_same_canonical_csr(fmt):
    from bnmtf_b200 import data
    rng = np.random.RandomState(1)
    D = np.where(rng.rand(30, 20) < 0.3, rng.rand(30, 20), np.nan)
    r, c = np.nonzero(~np.isnan(D))
    vals = D[r, c]
    vals[::7] = 0.0                                         # explicit zeros
    base = sp.coo_matrix((vals, (r, c)), shape=D.shape)
    A = sp.csr_array(base) if fmt == "csr_array" else base.asformat(fmt)
    if fmt in ("lil", "dok"):                               # these formats cannot store an explicit zero
        vals = vals.copy()
        vals[vals == 0] = 0.25
        base = sp.coo_matrix((vals, (r, c)), shape=D.shape)
        A = base.asformat(fmt)
    Rc, Mc, train = data.validate_sparse(A)
    assert Rc.nnz == r.size and train.all() and Mc.nnz == r.size
    ref = sp.csr_matrix(base)
    ref.sort_indices()
    np.testing.assert_array_equal(Rc.indptr, ref.indptr)
    np.testing.assert_array_equal(Rc.indices, ref.indices)
    np.testing.assert_array_equal(Rc.data, ref.data)


def test_unsorted_indices_are_canonicalised():
    from bnmtf_b200 import data
    A = sp.csr_matrix((np.array([2.0, 1.0, 0.0]), np.array([2, 0, 1]), np.array([0, 3])), shape=(1, 3))
    assert not A.has_sorted_indices
    Rc, _, _ = data.validate_sparse(A)
    np.testing.assert_array_equal(Rc.indices, [0, 1, 2])
    np.testing.assert_array_equal(Rc.data, [1.0, 0.0, 2.0])


def test_validation_rules():
    for cls in classes():
        dup = sp.coo_matrix((np.ones(3), ([0, 0, 1], [1, 1, 0])), shape=(2, 2))
        with pytest.raises(ValueError):
            cls(dup, None, 2, PRI)
        with pytest.raises(ValueError):
            cls(small(), sp.coo_matrix((np.ones(1), ([1], [2])), shape=(3, 3)), 2, PRI)     # (1, 2) is not stored in R
        with pytest.raises(ValueError):
            cls(small(), None, 2, PRI, distributed=True)
        with pytest.raises(AssertionError) as e:
            cls(small(), sp.coo_matrix((np.ones(1), ([0], [0])), shape=(3, 4)), 2, PRI)
        assert str(e.value) == "Input matrix R is not of the same size as the indicator matrix M: (3, 3) and (3, 4) respectively."
        M = sp.coo_matrix((np.ones(3), ([0, 0, 2], [0, 2, 0])), shape=(3, 3))        # row 1 has no training entry
        with pytest.raises(AssertionError) as e:
            cls(small(), M, 2, PRI)
        assert str(e.value) == "Fully unobserved row in R, row 1."
        R = sp.coo_matrix((np.ones(3), ([0, 1, 2], [0, 0, 1])), shape=(3, 3))
        with pytest.raises(AssertionError) as e:
            cls(R, None, 2, PRI)
        assert str(e.value) == "Fully unobserved column in R, column 2."
        M = sp.coo_matrix((np.array([1.0, 0.0, 1.0, 1.0, 1.0]), ([0, 0, 1, 2, 2], [0, 2, 1, 0, 2])), shape=(3, 3))
        m = cls(small(), M, 2, PRI)
        assert m.size_Omega == 4.0                          # a stored zero of M is not a training entry


def random_sparse(I, J, frac, seed):
    rng = np.random.RandomState(seed)
    Mfull = rng.rand(I, J) < frac
    Mfull[np.arange(I), rng.randint(0, J, I)] = True
    Mfull[rng.randint(0, I, J), np.arange(J)] = True
    r, c = np.nonzero(Mfull)
    vals = rng.exponential(1.0, r.size)
    vals[::11] = 0.0
    return sp.coo_matrix((vals, (r, c)), shape=(I, J)), Mfull


def test_csr_csc_and_plan_cover_every_entry_once():
    from bnmtf_b200.engine import csr_work_plan
    from bnmtf_b200 import data
    A, _ = random_sparse(300, 40, 0.3, 2)
    Rc, _, _ = data.validate_sparse(A.tocsr())
    C = Rc.tocsc()
    assert np.array_equal(C.toarray(), Rc.toarray()) and C.nnz == Rc.nnz
    for indptr in (Rc.indptr, C.indptr, np.array([0, 0, 5, 5, 37, 40], dtype=np.int64)):
        for chunk in (1, 4, 7, 64):
            p = csr_work_plan(indptr, chunk)
            rows = indptr.shape[0] - 1
            covered = np.zeros(int(indptr[-1]), dtype=int)
            seen_rows = np.zeros(rows, dtype=int)
            for b, r, s in zip(p["item_begin"], p["item_row"], p["item_slot"]):
                e = min(b + chunk, indptr[r + 1])
                assert indptr[r] <= b <= indptr[r + 1]
                covered[b:e] += 1
                seen_rows[r] += 1
            assert (covered == 1).all()
            assert (seen_rows >= 1).all()
            heavy = set(p["heavy_row"].tolist())
            assert heavy == {r for r in range(rows) if indptr[r + 1] - indptr[r] > chunk}
            for h, r in enumerate(p["heavy_row"]):
                slots = p["item_slot"][p["item_row"] == r]
                np.testing.assert_array_equal(slots, np.arange(p["heavy_first"][h], p["heavy_first"][h + 1]))
            assert (p["item_slot"][~np.isin(p["item_row"], p["heavy_row"])] == -1).all()
            assert p["n_slots"] == int(p["heavy_first"][-1])


def csr_stats_numpy(indptr, indices, data, Xp, Vp, chunk):
    """What bnmtf_csr_stats_f64 computes, restated: per work item the sums over its entries, the chunk partials of a heavy
    row added in chunk order.  -> RX (rows x KP), G (rows x KP x KP, full), SV (rows x KP)."""
    from bnmtf_b200.engine import csr_work_plan
    p = csr_work_plan(indptr, chunk)
    rows, KP = indptr.shape[0] - 1, Xp.shape[1]
    RX, G, SV = np.zeros((rows, KP)), np.zeros((rows, KP, KP)), np.zeros((rows, KP))
    parts = {}
    for b, r, s in zip(p["item_begin"], p["item_row"], p["item_slot"]):
        e = min(b + chunk, indptr[r + 1])
        X = Xp[indices[b:e]]
        part = (data[b:e] @ X, X.T @ X, Vp[indices[b:e]].sum(axis=0))
        if s < 0:
            RX[r], G[r], SV[r] = part
        else:
            parts.setdefault(r, []).append((s, part))
    for r, lst in parts.items():
        lst.sort(key=lambda t: t[0])
        acc = [x.copy() for x in lst[0][1]]
        for _, part in lst[1:]:
            for a, x in zip(acc, part):
                a += x
        RX[r], G[r], SV[r] = acc
    return RX, G, SV


@pytest.mark.parametrize("K", [3, 7, 8, 20])
def test_chunked_csr_statistics_equal_the_dense_masked_statistics_of_the_oracle(K):
    from oracle import bnmtf_oracle as orc
    from bnmtf_b200 import data
    A, _ = random_sparse(120, 90, 0.15, K)
    Rc, Mc, train = data.validate_sparse(A)
    R, M = Rc.toarray(), Mc.toarray()
    rng = np.random.RandomState(K)
    U, V, varV = rng.exponential(1.0, (120, K)), rng.exponential(1.0, (90, K)), rng.exponential(0.1, (90, K))
    KP = 8 * ((K + 1 + 7) // 8)
    Xp, Vp = np.zeros((90, KP)), np.zeros((90, KP))
    Xp[:, :K], Xp[:, K], Vp[:, :K] = V, 1.0, varV
    RX, G, SV = csr_stats_numpy(Rc.indptr, Rc.indices, Rc.data, Xp, Vp, chunk=5)
    # the dense masked statistics (bnmtf_stats_rx_f64 / bnmtf_stats_gram_f64 at polarity 1)
    np.testing.assert_allclose(RX, (M * R) @ Xp, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(G, np.einsum("ij,jk,jl->ikl", M, Xp, Xp), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(SV, M @ Vp, rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(G[:, K, K], M.sum(axis=1))          # slot (K, K): the count
    # ... and they reproduce the oracle's conditional parameters (bnmf_vb_optimised.py:189-191) for every column
    o = orc.OracleBNMF(R, M, K, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}, mode="vb")
    o.set_state(U, V, tau=2.5, varU=np.zeros_like(U), varV=varV)
    o.exptau = 2.5
    for k in range(K):
        tau_k, mu_k = o.column_params(k, "U")
        t = 2.5 * (G[:, k, k] + SV[:, k])
        s = RX[:, k] - (G[:, k, :K] * U).sum(axis=1) + G[:, k, k] * U[:, k]
        np.testing.assert_allclose(t, tau_k, rtol=1e-12)
        np.testing.assert_allclose((-0.1 + 2.5 * s) / t, mu_k, rtol=1e-9, atol=1e-12)


def test_sparse_predict_needs_a_pattern_inside_R():
    from bnmtf_b200 import data
    Rc, _, _ = data.validate_sparse(small())
    sel = data.sparse_selection(Rc, sp.coo_matrix((np.ones(2), ([0, 2], [2, 2])), shape=(3, 3)))
    np.testing.assert_array_equal(sel, [False, True, False, False, True])
    with pytest.raises(ValueError):
        data.sparse_selection(Rc, sp.coo_matrix((np.ones(1), ([1], [0])), shape=(3, 3)))
    with pytest.raises(ValueError):
        data.sparse_selection(Rc, np.ones((3, 3)))
